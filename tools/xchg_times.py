"""Where the strip exchange spends its time (run under torchrun, N >= 2): strip build alone, build + exchange one
at a time, the exchange alone (events around gndt_xchg_run)."""
import ctypes as C, json, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch, torch.distributed as dist
import bench
from grid_ndt_b200._lib import lib
from grid_ndt_b200.builder import _check
from grid_ndt_b200.tiles import TiledTwoDmap
rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local); dev = torch.device("cuda", local)
dist.init_process_group("nccl", device_id=dev)
cloud = torch.from_numpy(bench.make_cloud(rank)).cuda()
origin = [float(np.float32(0.5 * bench.SCENE_W + 0.013)), float(np.float32(40.007)), 1.0]
gather = tuple(os.environ.get("GATHER", "slopes,columns").split(","))
tm = TiledTwoDmap(0.2, 0.1, 0.08, rank, world, device=local, gather=gather, capacity=int(0.08 * 1e7 * world) + 1_000_000)
m, L = tm.map, lib()
def timed(fn, n=20):
    for _ in range(3): fn()
    dist.barrier(); torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n): fn()
    e1.record(); torch.cuda.synchronize()
    t = torch.tensor([e0.elapsed_time(e1) / n], device=dev); dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())
m.setCloudFirst(origin)
def build_only():
    m.uniformDivision(cloud); m.create2DMap("slope")
def build_xchg():
    tm.build(cloud, "slope", origin=origin, cuts=None, filter_points=False)
def xchg_only():
    _check(m._h, L.gndt_xchg_run(m._h, torch.cuda.current_stream().cuda_stream))
res = {"world": world, "gather": gather,
       "build_ms": timed(build_only), "build_xchg_ms": timed(build_xchg)}
build_only(); torch.cuda.synchronize(); dist.barrier()
res["xchg_only_ms"] = timed(xchg_only)
if rank == 0: print(json.dumps(res), flush=True)
tm.close(); dist.barrier(); dist.destroy_process_group()
