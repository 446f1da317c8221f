"""Diagnosis: pipelined throughput of TiledTwoDmap (DEPTH builds in flight, default 3) with the exchange transport
TRANSPORT ("sm" or "ce").  Run under torchrun; one setting per process."""
import json, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch, torch.distributed as dist
import bench
from grid_ndt_b200.tiles import TiledTwoDmap
rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local); dev = torch.device("cuda", local)
dist.init_process_group("nccl", device_id=dev)
cloud = torch.from_numpy(bench.make_cloud(rank)).cuda()
origin = [float(np.float32(0.5 * bench.SCENE_W + 0.013)), float(np.float32(40.007)), 1.0]
depth = int(os.environ.get("DEPTH", "3"))
tm = TiledTwoDmap(0.2, 0.1, 0.08, rank, world, device=local, depth=depth, transport=os.environ.get("TRANSPORT"), gather=("slopes", "columns"), capacity=int(0.08 * 1e7 * world) + 1_000_000)
build_ms = []
def run(k):
    ahead = 0
    for i in range(k):
        while ahead < min(k, i + tm.depth):
            tm.submit(cloud, "slope", origin=origin, cuts=None, filter_points=False); ahead += 1
        s = tm.wait_oldest()
        build_ms.append(s.build_start.elapsed_time(s.build_done))
    tm.join()
run(6); dist.barrier(); torch.cuda.synchronize()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record(); run(30); e1.record(); torch.cuda.synchronize()
t = torch.tensor([e0.elapsed_time(e1) / 30], device=dev); dist.all_reduce(t, op=dist.ReduceOp.MAX)
bm = torch.zeros(world, device=dev); bm[rank] = float(np.mean(build_ms[-30:])); dist.all_reduce(bm)
if rank == 0: print(json.dumps({"world": world, "depth": depth, "transport": tm.transport, "ms_per_step": round(float(t.item()), 4), "build_ms_per_rank": [round(float(x), 3) for x in bm.tolist()]}), flush=True)
dist.barrier(); dist.destroy_process_group()
