#!/usr/bin/env python
"""bench.py — NDT map-build throughput (BASELINE.json metric) on N B200s of one node.

  python bench.py [--gpus N] [--steps K] [--warmup W]            our CUDA path
  python bench.py --impl reference [--gpus N] [--steps K] ...    the reference's own CPU code

A "step" is one complete map build (bounds -> partition -> fit -> labels -> edges) of one
synthetic cloud.  N = 1: BASELINE.json configs[1] (cfg2: 10 M points, multi-level bridge /
underpass scene, 0.2 m cells).  N > 1: one x strip per GPU, each strip one cfg2 scene
(weak scaling: 10 M points per GPU); the thin halo rows and the gather of the finished
Slope + Cell tables (what the host planner reads) go through peer-mapped memory inside
libgndt.so (csrc/gndt_exchange.cuh), inside the timed region.  NCCL only carries the
barrier / max-over-ranks of the timing itself.

`value`         : points/s, device-timed with CUDA events, inputs resident in HBM, max over
                  ranks, K back-to-back builds with two (N > 1: three) in flight on separate
                  streams.  `value_latency` / `serial_ms_per_step`: one build at a time.
`e2e`           : the same metric through the public TwoDmap call with PINNED HOST input, the
                  host->device copy of the cloud and the device->host copy of the result
                  tables inside the timed region, every step (N > 1: every rank uploads its
                  cloud, rank 0 reads back the gathered Slope + Cell tables of the WHOLE map).
`roofline`      : algorithmic bytes of one build (16 B per point read once + 96 B per voxel
                  record written once, SURVEY.md §8(d)) / device time of one build alone,
                  against the measured HBM copy bandwidth in MEASURED_PEAKS.json.
N > 1 adds, outside the timed region: `parity` (a 2 M-point strip build + exchange held to
the full parity bar against the oracle on rank 0; the run fails on any unexplained mismatch)
and `target_cfg3` (the north-star case: ONE 50 M-point cloud at 0.1 m cells, strong-scaled
over the N strips, both input conventions).

--dump-outputs DIR (N = 1): after the run, the voxel, slope and column tables of the last timed
step, one DIR/<table>_<field>.npy per field (float fields float32, integer fields float64, both
exact), DIR/<table>_rows.npy (the table rows written) and DIR/counts.npy.  Tables longer than
DUMP_ROWS rows are written as a seeded sample of rows that depends only on the table's length:
two runs whose tables have the same length get the same rows (counts.npy tells when they do
not).  The input cloud is seeded, so two builds of the project can be compared output for output.
"""
import argparse
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

CFG = "cfg2"
POINTS_PER_GPU = 10_000_000
GRID_LEN, Z_LEN, INTERVAL = 0.2, 0.1, 0.08
SCENE_W = 120.0
DEPTH = int(os.environ.get("GNDT_BENCH_DEPTH", "3"))  # N > 1: builds in flight
REF_STEP_POINTS = 1_000_000      # --impl reference: points per timed step (bounded sample)
CPU_BASELINE_POINTS = 4_000_000  # cpu_baseline leg of the default run
TARGET_POINTS = int(os.environ.get("GNDT_BENCH_TARGET_POINTS", "50000000"))  # north-star cloud (N > 1); 0 disables
WORKLOAD = "cfg2 multi-level bridge/underpass scene, 10M points per GPU, 0.2 m cells, z 0.1 m, slope_interval 0.08, demand slope (BASELINE configs[1])"
DUMP_ROWS, DUMP_SEED = 200_000, 20260100  # --dump-outputs: rows per table (at most 55 MB in all)


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "MEASURED_PEAKS.json (device copy, measured)"
    except Exception:
        return 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md; MEASURED_PEAKS.json absent)"


def bind_to_gpu_numa_node(index):
    """Run this process (and first-touch its pinned buffers) on the NUMA node the GPU hangs off:
    with 8 ranks on one box, host buffers on the wrong socket cross the inter-socket link on every
    upload.  Returns a short description for the JSON line."""
    try:
        import pynvml
        pynvml.nvmlInit()
        bus = pynvml.nvmlDeviceGetPciInfo(pynvml.nvmlDeviceGetHandleByIndex(index)).busId
        bus = (bus.decode() if isinstance(bus, bytes) else bus).lower()
        if len(bus.split(":")[0]) == 8:
            bus = bus[4:]
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read())
        if node < 0:
            return "numa node unknown (single node or virtualised)"
        cpus = []
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus += range(int(lo), int(hi or lo) + 1)
        allowed = sorted(set(cpus) & os.sched_getaffinity(0))
        if allowed:
            os.sched_setaffinity(0, allowed)
            return f"bound to numa node {node} ({len(allowed)} cpus)"
        return f"numa node {node}: no allowed cpus, not bound"
    except Exception as e:  # best effort: never fail the bench over affinity
        return f"not bound ({type(e).__name__})"


class ClockSampler:
    """Polls SM clock and throttle reasons through NVML while the timed region runs."""

    def __init__(self, index):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thr = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _loop(self):
        nv = self.nv
        names = {}
        for k in dir(nv):
            if k.startswith("nvmlClocksEventReason") or k.startswith("nvmlClocksThrottleReason"):
                v = getattr(nv, k)
                if isinstance(v, int) and v:
                    names[v] = k.replace("nvmlClocksEventReason", "").replace("nvmlClocksThrottleReason", "")
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, nm in names.items():
                    if r & bit and bin(bit).count("1") == 1:
                        self.reasons.add(nm)
            except Exception:
                pass
            time.sleep(0.002)

    def __enter__(self):
        if self.nv:
            self._thr = threading.Thread(target=self._loop, daemon=True)
            self._thr.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self._thr:
            self._thr.join()

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["unavailable"]}
        reasons = sorted(r for r in self.reasons if r not in ("GpuIdle", "None", "ApplicationsClocksSetting"))
        return {"sm_mhz": statistics.median(self.samples), "sm_max_mhz": self.max_mhz, "reasons": reasons, "samples": len(self.samples)}


def make_cloud(rank):
    """cfg2 scene for strip `rank`, shifted by rank * 120 m in x (common frame)."""
    from grid_ndt_b200 import synthetic
    cloud = synthetic.cfg2(POINTS_PER_GPU)
    if rank:
        # the whole scene moves, its (0,0,0) padding included: every strip keeps one pathologically heavy voxel at
        # ITS sensor origin and the same extent (leaving the padding at the global origin stretched the bounding
        # box of every strip but the first over the whole map, costing those strips a partition pass)
        cloud[:, 0] += np.float32(SCENE_W * rank)
    return cloud


def dump_outputs(out_dir, m):
    """The result tables of the build held by TwoDmap `m` -> out_dir/<table>_<field>.npy."""
    from grid_ndt_b200._abi import Counts
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"counts": np.array([m.counts()[k] for k, _ in Counts._fields_], np.float64)}
    for table in ("voxels", "slopes", "columns"):
        t = getattr(m, table)
        rows = np.arange(len(t))
        if len(t) > DUMP_ROWS:
            rows = np.sort(np.random.default_rng(DUMP_SEED).choice(len(t), DUMP_ROWS, replace=False))
        arrays[f"{table}_rows"] = rows.astype(np.float64)
        for field in t.dtype.names:
            if field != "reserved":
                a = t[field][rows]
                arrays[f"{table}_{field}"] = a.astype(np.float32 if a.dtype.kind == "f" else np.float64)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)
    return sum(a.nbytes for a in arrays.values())


def run_reference(args):
    """The reference's own CPU implementation of the path (oracle/_ref: src/receiver.cpp +
    include/map2D.h compiled against inert shims), single-threaded like its initial-build
    loop (the OpenMP pragma at src/receiver.cpp:149 is commented out).  `value` counts only the
    reference's own two stage timers ("division time" + "calculate time", src/receiver.cpp:148-162):
    the harness's copy into the reference containers and the teardown of its maps are excluded."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    from grid_ndt_b200 import synthetic
    from grid_ndt_b200._abi import default_params
    from oracle import oracle as O

    kind = "reference" if os.path.exists(O.REF_SO) else "port"
    fn = O.ref_build if kind == "reference" else (lambda c, p: O.oracle_build(c, p, "faithful32"))
    cloud = synthetic.cfg2(POINTS_PER_GPU)[:REF_STEP_POINTS]
    p = default_params(GRID_LEN, Z_LEN, INTERVAL)
    for _ in range(args.warmup):
        fn(cloud[: REF_STEP_POINTS // 8], p)
    stage_s, t0 = 0.0, time.perf_counter()
    for _ in range(args.steps):
        r = fn(cloud, p)
        stage_s += r.division_s + r.calculate_s
    wall = time.perf_counter() - t0
    value = REF_STEP_POINTS * args.steps / stage_s
    sample = (f"first {REF_STEP_POINTS} points of the 10M-point cfg2 cloud per step (the GPU arm builds all 10M per step), {kind} build; "
              f"value = points / (division + calculate timers of the reference, {stage_s / args.steps:.2f} s per step); wall incl. harness {wall / args.steps:.2f} s per step")
    line = {
        "impl": "reference", "metric": "ndt_map_build_points_per_sec", "value": value, "unit": "points/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * stage_s / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "points_per_step": REF_STEP_POINTS,
                   "subsample": "the CPU arm times a 1M-point prefix of the same cloud per step (10M points take about 20 s per step on one core); points/s is size-normalised"},
        "cpu_baseline": {"value": value, "unit": "points/s", "cores": 1, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": "points/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "wall_points_per_s_incl_harness": REF_STEP_POINTS * args.steps / wall,
        "gpu_launches": 0,
    }
    args.json_out.write(json.dumps(line) + "\n")
    args.json_out.flush()
    return 0


def multi_gpu_parity(rank, world, local, transport=None):
    """Outside the timed region: one 2 M-point cloud cut into `world` strips, built, exchanged,
    and (rank 0) compared with the oracle to the full parity bar (tests/parity.py)."""
    import torch
    from grid_ndt_b200 import synthetic
    from grid_ndt_b200._abi import default_params
    from grid_ndt_b200.tiles import TiledTwoDmap
    cloud = synthetic.cfg2(2_000_000, scale=0.2 ** 0.5)
    origin = [float(v) for v in cloud[0, :3]]
    dev_cloud = torch.from_numpy(cloud).cuda()
    tm = TiledTwoDmap(GRID_LEN, Z_LEN, INTERVAL, rank, world, device=local, capacity=3_000_000, transport=transport)
    cuts = tm.plan(dev_cloud, origin=origin)
    tm.build(dev_cloud, "slope", origin=origin, cuts=cuts, filter_points=True)
    out = None
    if rank == 0:
        from oracle import oracle as O
        from tests import parity
        p = default_params(GRID_LEN, Z_LEN, INTERVAL, origin=origin, origin_is_first_point=0)
        o32, o64 = O.oracle_build(cloud, p, "faithful32"), O.oracle_build(cloud, p, "truth64")
        rep = parity.compare_gathered(tm.gathered_numpy("voxels"), tm.gathered_numpy("columns"), tm.gathered_numpy("slopes"), o32, o64, p)
        unexplained = (rep.get("label_mismatch", 0) - rep.get("label_mismatch_agreeing_with_truth64", 0) - rep.get("label_mismatch_threshold_adjacent", 0)
                       + rep.get("reach_mismatch", 0) - rep.get("reach_mismatch_agreeing_with_truth64", 0) - rep.get("reach_mismatch_threshold_adjacent", 0))
        out = {"points": int(cloud.shape[0]), "strips": world, "voxels": int(len(o32.voxels)), "ok": bool(rep["ok"]),
               "label_mismatch": rep.get("label_mismatch"), "reach_mismatch": rep.get("reach_mismatch"), "unexplained": int(unexplained) if rep["ok"] else -1,
               "exact_fields": "sx sy sz count first_index column slope: bit-exact" if rep["ok"] else rep["fail"],
               "mean_max_rel_err": rep.get("mean_max_rel_err"), "scatter_max_rel_err": rep.get("scatter_max_rel_err"), "evals_max_rel_err": rep.get("evals_max_rel_err")}
    else:
        tm.synchronize()
    tm.close()
    del dev_cloud
    torch.cuda.empty_cache()
    return out


def target_cfg3(rank, world, local, dev, peak, transport=None):
    """North star: ONE cloud (cfg3 terrain, 50 M points, 0.1 m cells) strong-scaled over the N
    strips, whole map (Slope + Cell tables) gathered on every GPU; cloud resident in HBM."""
    import torch
    import torch.distributed as dist
    from grid_ndt_b200 import synthetic
    from grid_ndt_b200.tiles import TiledTwoDmap
    n = TARGET_POINTS
    cloud = synthetic.cfg3(n, extent=224.0 * (n / 50e6) ** 0.5)  # same seed on every rank
    origin = [float(v) for v in cloud[0, :3]]
    full = torch.from_numpy(cloud).cuda()
    tm = TiledTwoDmap(0.1, 0.1, INTERVAL, rank, world, device=local, halo_records=65536, gather=("slopes", "columns"),
                      capacity=int(0.2 * n) + 1_000_000, transport=transport)
    cuts = tm.plan(full, origin=origin)
    rows = {}
    for mode in ("full", "share"):
        if mode == "full":
            src, filt = full, True
        else:  # this rank's strip only: the reference's x index (map2D.h:965-970) evaluated on the host
            d = cloud[:, 0] - np.float32(origin[0])
            k = np.maximum(np.ceil((np.abs(d) / np.float32(0.1)).astype(np.float32)), 1).astype(np.int64)
            cx = np.where(cloud[:, 0] > np.float32(origin[0]), k - 1, -k)
            src, filt = torch.from_numpy(np.ascontiguousarray(cloud[(cx >= cuts[rank]) & (cx < cuts[rank + 1])])).cuda(), False
        fn = (lambda: tm.build(src, "slope", origin=origin, cuts=cuts, filter_points=filt))
        for _ in range(2):
            fn()
        dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        steps = 5
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        dist.barrier()
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1) / steps], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
        total_vox = int(tm.offsets[-1])
        b_alg = 16.0 * n + 96.0 * total_vox
        rows[mode] = {"ms_per_build": ms, "points_per_s": n / ms * 1e3, "frac_of_aggregate_peak": b_alg / ms / 1e6 / (peak * world),
                      "voxels": total_vox, "meets_10ms": bool(ms < 10.0)}
        del src
    tm.close()
    del full
    torch.cuda.empty_cache()
    rows["what"] = (f"ONE cfg3 terrain cloud, {n // 1_000_000}M points, 0.1 m cells, x strips over {world} GPUs, Slope + Cell tables of the whole map "
                    "gathered on every GPU through peer-mapped memory; 'full': every GPU holds the whole cloud and filters its strip in the first pass, "
                    "'share': every GPU holds only its strip's points; target < 10 ms on 8 GPUs at >= 60 % of the aggregate HBM roofline")
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="N > 1: skip the parity and target_cfg3 legs")
    ap.add_argument("--dump-outputs", metavar="DIR", help="N = 1: write the result tables of the last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or int(os.environ.get("WORLD_SIZE", "1")) > 1):
        ap.error("--dump-outputs writes the tables of a single-GPU build of our path: run it with --impl ours and one process")
    args.warmup = max(args.warmup, 3)
    # stdout carries exactly ONE line, the JSON: everything else any library writes to fd 1
    # (NCCL's version banner, for one) is sent to stderr for the whole run
    sys.stdout.flush()
    json_out = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    args.json_out = json_out
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    from grid_ndt_b200 import TwoDmap

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: there is no CPU fallback for the product path")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa = bind_to_gpu_numa_node(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    cloud = make_cloud(rank)
    n_pts = cloud.shape[0]
    host = torch.from_numpy(cloud).pin_memory()
    resident = host.to(dev)
    origin = [float(np.float32(0.5 * SCENE_W + 0.013)), float(np.float32(40.007)), 1.0]  # cfg2's designated first point

    if world > 1:
        from grid_ndt_b200.tiles import TiledTwoDmap
        cap = int(0.08 * n_pts * world) + 1_000_000  # voxels of the whole map (cfg2: 0.055 per point)
        gather = ("slopes", "columns")              # what the host planner reads (Cell / Slope, map2D.h:136-187)
        # DEPTH builders deep: the NVLink gather of build i overlaps the SM work of the next builds
        pair, parked = {}, []

        def make(transport):
            pair["tmp"] = TiledTwoDmap(GRID_LEN, Z_LEN, INTERVAL, rank, world, device=local, depth=DEPTH, gather=gather, capacity=cap, transport=transport)
            pair["tm"] = TiledTwoDmap(GRID_LEN, Z_LEN, INTERVAL, rank, world, device=local, depth=1, gather=gather, capacity=cap, transport=transport)  # one at a time

        def park():
            """Set the current builders aside WITHOUT freeing them: their exchange buffers are mapped by the peers
            (an exported buffer must outlive the peers' mappings), so everything is closed together at the end."""
            for k in ("tmp", "tm"):
                if k in pair:
                    parked.append(pair.pop(k))

        def step(src):
            return pair["tm"].build(src, "slope", origin=origin, cuts=None, filter_points=False)

        def run_steps(src, k):
            tmp = pair["tmp"]
            n_launch = 0
            ahead = 0
            for i in range(k):
                while ahead < min(k, i + tmp.depth):  # keep `depth` builds in flight
                    tmp.submit(src, "slope", origin=origin, cuts=None, filter_points=False)
                    ahead += 1
                tmp.collect()
                n_launch += tmp.last_map.launch_count()
            tmp.join()
            return n_launch

        def probe(transport, k=12):
            """ms per pipelined step with this transport of the strip records (max over ranks), inf if any rank failed"""
            ok, ms, why = 1.0, float("inf"), ""
            try:
                make(transport)
                run_steps(resident, 4)
                step(resident)
                torch.cuda.synchronize()  # no collective inside the try: a rank that fails must still meet the others below
                p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                p0.record(); run_steps(resident, k); p1.record()
                torch.cuda.synchronize()
                ms = p0.elapsed_time(p1) / k
            except Exception as e:  # e.g. the exchange watchdog: fall back to the other transport on EVERY rank
                ok, why = 0.0, f"{type(e).__name__}: {e}"
                print(f"[rank {rank}] transport {transport} failed: {why}", file=sys.stderr, flush=True)
            t = torch.tensor([-ok, ms if ok else 0.0], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t[1].item()) if t[0].item() == -1.0 else float("inf")

        # which engine carries the strip records to the peers: the copy engines ("ce") or an SM kernel ("sm").
        # Both are timed during warm-up; the faster one runs the timed region (GNDT_BENCH_TRANSPORT pins it).
        forced = os.environ.get("GNDT_BENCH_TRANSPORT")
        probes = {}
        if forced:
            make(forced)
            chosen = forced
        else:
            kept = {}
            for tr in ("sm", "ce"):
                probes[tr] = probe(tr)
                kept[tr] = dict(pair)
                park()
            if probes["ce"] == probes["sm"] == float("inf"):
                raise RuntimeError("both exchange transports failed")
            chosen = "ce" if probes["ce"] <= probes["sm"] else "sm"
            pair.update(kept[chosen])
        m = pair["tm"].map
    else:
        from grid_ndt_b200.pipeline import CloudPipeline
        m = TwoDmap(GRID_LEN, Z_LEN, device=local)  # one build at a time: stage times, latency, e2e serial
        m.setInterval(INTERVAL)
        # throughput: two builds in flight on two streams (a second build fills the SMs left idle
        # by the partial last wave of every kernel and by the tiny kernels of the first)
        flight = CloudPipeline(GRID_LEN, Z_LEN, INTERVAL, "slope", depth=2, device=local)
        last = {}  # the builder of the last step run_steps submitted (flight is not used after the timed region)

        def step(src):
            m.chatterCallback(src, "slope")

        def run_steps(src, k):
            n_launch = 0
            for _ in range(k):
                if flight.pending == flight.depth:
                    n_launch += flight.release().launch_count()
                flight.submit(src)
            while flight.pending:
                last["map"] = flight.release()
                n_launch += last["map"].launch_count()
            flight.join()
            return n_launch

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(v):
        if world > 1:
            t = torch.tensor([v], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())
        return v

    run_steps(resident, args.warmup)
    step(resident)
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local) as clk:
        barrier()
        ev0.record()
        launches = run_steps(resident, args.steps)
        ev1.record()
        barrier()
    ms_per_step = max_over_ranks(ev0.elapsed_time(ev1)) / args.steps
    total_pts = n_pts * world
    value = total_pts / (ms_per_step * 1e-3)
    # one build at a time (latency of a single cloud), same events, outside the headline region
    barrier()
    es0, es1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n_serial = max(3, min(args.steps, 10))
    es0.record()
    for _ in range(n_serial):
        step(resident)
    es1.record()
    barrier()
    serial_ms = max_over_ranks(es0.elapsed_time(es1)) / n_serial
    # stage split of one build alone (stage events cost a little: kept out of the numbers above)
    m.stage_timing(True)
    step(resident)
    barrier()
    counts = m.counts()
    stages = m.stage_ms()
    layout = m.key_layout()
    m.stage_timing(False)

    # ---- end to end: pinned host cloud in, result tables out (into pinned host buffers), every step
    m.pin_results(True)
    if world > 1:
        # The host planner is one consumer: the whole map must reach ONE host buffer.  Every rank copies ITS strip
        # of the gathered Slope + Cell tables (indices already global) into a buffer shared by all ranks (POSIX
        # shared memory, page-locked in every process), so the read-back uses all N PCIe links instead of rank 0's.
        from multiprocessing import shared_memory
        cap_rec = cap
        shm_bytes = cap_rec * (48 + 32)
        name = [None]
        if rank == 0:
            shm = shared_memory.SharedMemory(create=True, size=shm_bytes)
            name[0] = shm.name
        dist.broadcast_object_list(name, src=0)
        if rank != 0:
            shm = shared_memory.SharedMemory(name=name[0])
        host_map = torch.from_numpy(np.ndarray((shm_bytes,), np.uint8, buffer=shm.buf))
        assert int(torch.cuda.cudart().cudaHostRegister(host_map.data_ptr(), shm_bytes, 0)) == 0
        col_base = cap_rec * 48

        def read_back(g):
            """this rank's strip of the gathered tables -> the shared host map; returns the bytes it moved"""
            sc = g.strip_counts
            s0, s1 = int(sc[:rank, 2].sum()) * 48, int(sc[:rank + 1, 2].sum()) * 48
            c0, c1 = int(sc[:rank, 1].sum()) * 32, int(sc[:rank + 1, 1].sum()) * 32
            host_map[s0:s1].copy_(g.slopes.reshape(-1)[s0:s1], non_blocking=True)
            host_map[col_base + c0: col_base + c1].copy_(g.columns.reshape(-1)[c0:c1], non_blocking=True)
            torch.cuda.current_stream().synchronize()
            return (s1 - s0) + (c1 - c0)

        def e2e_step():
            return read_back(step(host))
    else:
        def e2e_step():
            step(host)
            v, s, c = m.voxels, m.slopes, m.columns
            return v.nbytes + s.nbytes + c.nbytes

    def wall(fn, n):
        barrier()
        t0 = time.perf_counter()
        fn(n)
        barrier()
        return max_over_ranks((time.perf_counter() - t0) / n)

    d2h = 0
    for _ in range(2):
        d2h = e2e_step()
    n_e2e = max(3, min(args.steps, 10))
    serial_s = wall(lambda n: [e2e_step() for _ in range(n)], n_e2e)
    e2e_s, e2e_mode = serial_s, "one build at a time: H2D -> kernels (+ peer-memory exchange at N>1) -> D2H"
    if world == 1:
        # the same call, two builders deep: the upload of cloud i+1 overlaps the build and
        # read-back of cloud i (grid_ndt_b200.pipeline.CloudPipeline).  Every step still
        # uploads its whole cloud and reads back all three tables inside the timed region.
        from grid_ndt_b200.pipeline import CloudPipeline
        pipe = CloudPipeline(GRID_LEN, Z_LEN, INTERVAL, "slope", depth=2, device=local)

        def piped(n):
            pipe.submit(host)
            for i in range(n):
                if i + 1 < n:
                    pipe.submit(host)
                r = pipe.collect()
                assert r["voxels"].nbytes + r["slopes"].nbytes + r["columns"].nbytes == d2h
        piped(3)
        e2e_s = wall(piped, n_e2e)
        e2e_mode = "CloudPipeline depth 2: H2D of cloud i+1 overlaps kernels + D2H of cloud i"
        pipe.close()
    else:
        tmp = pair["tmp"]

        def piped(n):
            tmp.submit(host, "slope", origin=origin, cuts=None, filter_points=False)
            for i in range(n):
                if i + 1 < n:
                    tmp.submit(host, "slope", origin=origin, cuts=None, filter_points=False)
                got = read_back(tmp.collect())
                assert got == d2h, (got, d2h)
            tmp.synchronize()
        piped(3)
        e2e_s = wall(piped, n_e2e)
        e2e_mode = (f"TiledTwoDmap depth {tmp.depth}, host input on every rank: H2D of cloud i+1 overlaps the exchange of cloud i; the gathered Slope + Cell "
                    "tables of the WHOLE map (the host planner's input) land in one host buffer shared by all ranks, each rank copying its own strip "
                    "over its own PCIe link; d2h_bytes_per_step is the whole map")
    e2e_value = total_pts / e2e_s
    if world > 1:
        t = torch.tensor([float(d2h)], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        d2h = int(t.item())
        torch.cuda.cudart().cudaHostUnregister(host_map.data_ptr())
        del host_map
        shm.close()
        if rank == 0:
            shm.unlink()

    peak, peak_src = measured_peak()
    v_tab = counts["n_voxels"]
    b_alg = 16.0 * n_pts + 96.0 * v_tab            # per GPU per build (SURVEY §8(d))
    # device time of one build alone: N = 1 the serial loop above (events around back-to-back single builds, no
    # stage events inside); N > 1 the library's start/end events of this rank's strip build (excludes the exchange)
    t_build_ms = serial_ms if world == 1 else stages["total"]
    achieved = b_alg / (t_build_ms * 1e-3) / 1e9
    traffic = None
    tp = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.exists(tp):
        try:
            traffic = json.load(open(tp)).get("build_dram_bytes")
        except Exception:
            traffic = None

    n_pass = max(1, layout["passes"])
    pass_ms = stages["sort"] / n_pass
    pass_bytes = 32.0 * n_pts  # every point read once and written once per pass
    dominant = {"name": "sort_pass_kernel", "launches_per_build": n_pass, "share_of_build": stages["sort"] / stages["total"],
                "algorithmic_bytes_per_launch": pass_bytes, "avg_launch_ms": pass_ms,
                "achieved": pass_bytes / (pass_ms * 1e-3) / 1e9, "frac": pass_bytes / (pass_ms * 1e-3) / 1e9 / peak,
                "note": "the same memory pattern with no other work runs at 4.9 TB/s (tools/micro/scatter_pattern.cu, 65 us)"}

    line = {
        "metric": "ndt_map_build_points_per_sec", "value": value, "unit": "points/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step,
        "ms_per_10M_points": ms_per_step * 1e7 / total_pts, "serial_ms_per_step": serial_ms,
        "value_latency": total_pts / (serial_ms * 1e-3),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD,
                   "points_per_gpu": n_pts, "voxels_per_gpu": v_tab, "columns_per_gpu": counts["n_columns"], "slopes_per_gpu": counts["n_slopes"],
                   "l2": "inputs (160 MB) and work buffers (320 MB) exceed the 126 MB L2; no explicit flush",
                   "parallelism": (f"x-strips x{world}: halo rows + gather of the Slope and Cell tables through peer-mapped memory over NVLink (no NCCL on the data path); "
                                   if world > 1 else "single GPU; ")
                                  + (f"{DEPTH if world > 1 else 2} builds in flight on separate streams for `value`; value_latency / serial_ms_per_step = one build at a time"),
                   "host": numa,
                   **({"exchange": {"transport": chosen, "what": "ce = strip records carried to the peers by the copy engines (one 256-byte host round trip per build, "
                                    "hidden behind the builds queued after it); sm = pushed by an SM kernel (no host round trip). Both timed during warm-up, the faster one kept",
                                    "probe_ms_per_step": {k: (None if v == float("inf") else v) for k, v in probes.items()}}} if world > 1 else {})},
        "stage_ms": stages,
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": traffic, "algorithmic_bytes": b_alg, "kernel_ms": t_build_ms,
                     "dominant_kernel": dominant,
                     "achieved_in_flight": (b_alg / (ms_per_step * 1e-3) / 1e9) if world == 1 else None,
                     "what": "whole build (all kernels of one step) on one GPU, one build at a time: (16 B x points + 96 B x voxels) / "
                             "device time of the build (library start/end events); achieved_in_flight = the same bytes / ms_per_step of the timed "
                             "region (two builds in flight); peak = " + peak_src},
        "e2e": {"value": e2e_value, "unit": "points/s", "h2d_bytes_per_step": int(n_pts * 16 * world), "d2h_bytes_per_step": int(d2h),
                "ms_per_step": e2e_s * 1e3, "mode": e2e_mode, "serial_ms_per_step": serial_s * 1e3,
                "h2d_gbs_per_gpu_if_copy_bound": n_pts * 16 / e2e_s / 1e9},
        "gpu_launches": launches,
        "clocks": clk.summary(),
    }
    if world > 1 and not args.no_extras:
        par = multi_gpu_parity(rank, world, local, chosen)  # the transport that ran the timed region
        bad = torch.tensor([0 if (par is None or (par["ok"] and par["unexplained"] == 0)) else 1], device=dev)
        dist.all_reduce(bad, op=dist.ReduceOp.MAX)
        line["parity"] = par
        if int(bad.item()):
            if rank == 0:
                sys.stderr.write("multi-GPU parity FAILED: " + json.dumps(par, default=str) + "\n")
            dist.destroy_process_group()
            return 1
        if TARGET_POINTS:
            line["target_cfg3"] = target_cfg3(rank, world, local, dev, peak, chosen)
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        from grid_ndt_b200._abi import default_params
        from oracle import oracle as O
        kind = "reference" if os.path.exists(O.REF_SO) else "port"
        fn = O.ref_build if kind == "reference" else (lambda c, p: O.oracle_build(c, p, "faithful32"))
        sample = cloud[:CPU_BASELINE_POINTS]
        t0 = time.perf_counter()
        r = fn(sample, default_params(GRID_LEN, Z_LEN, INTERVAL))
        dt = time.perf_counter() - t0
        line["cpu_baseline"] = {"value": CPU_BASELINE_POINTS / (r.division_s + r.calculate_s), "unit": "points/s", "cores": 1, "kind": kind,
                                "sample": f"first {CPU_BASELINE_POINTS} points of the same 10M cloud, one build: division {r.division_s:.1f} s + calculate {r.calculate_s:.1f} s "
                                          f"on the reference's own timers ({dt:.1f} s wall incl. the harness); single thread like the reference's initial-build loop",
                                "host_cores_available": os.cpu_count()}
    if rank == 0:
        args.json_out.write(json.dumps(line) + "\n")
        args.json_out.flush()
    if args.dump_outputs:
        nbytes = dump_outputs(args.dump_outputs, last["map"])
        print(f"outputs of the last timed step: {nbytes / 1e6:.1f} MB in {args.dump_outputs}", file=sys.stderr)
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
