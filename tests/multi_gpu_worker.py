"""torchrun worker for the N>1 GPU tests: every rank sees the whole cloud, plans the same
balanced x strips, builds its strip, and the strips are exchanged through peer-mapped memory
(default) or NCCL point-to-point.  The gathered map is held to the SAME bar as a single-GPU
build (tests/parity.compare against both oracle modes: integer fields bit-exact, floats within
1e-5, every label / reach mismatch proven threshold-adjacent) and must equal the untiled GPU
build byte for byte."""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np
import torch
import torch.distributed as dist

from grid_ndt_b200 import TwoDmap, _abi, synthetic
from grid_ndt_b200._abi import default_params
from grid_ndt_b200.tiles import TiledTwoDmap
from tests import parity


def untiled(cloud, origin):
    m = TwoDmap(0.2, 0.1)
    m.setInterval(0.08)
    m.setCloudFirst(origin)
    m.uniformDivision(cloud)
    m.create2DMap("slope")
    out = (m.voxels.copy(), m.slopes.copy(), m.columns.copy())
    m.close()
    return out


def same_table(tag, got, ref, exact=False):
    """Strips vs the untiled build of the same GPU code: integer fields, labels and indices
    identical; floats identical except for voxels whose points straddle a reduce tile, where the
    pairwise (Chan) merge of the binary64 partial sums associates differently because the tile
    boundaries fall elsewhere (last-bit noise: <= 1e-6 relative).  exact=True: bytes."""
    if got.tobytes() == ref.tobytes():
        return
    msg = [f"{tag}: {len(got)} records vs {len(ref)}"]
    ok = len(got) == len(ref) and not exact
    if len(got) == len(ref):
        for f in got.dtype.names:
            a, b = got[f], ref[f]
            bad = (a != b) if a.ndim == 1 else (a != b).any(axis=1)
            if not bad.any():
                continue
            i = int(np.nonzero(bad)[0][0])
            if a.dtype.kind == "f" and not exact:
                scale = np.maximum(np.abs(b).max(axis=-1) if b.ndim > 1 else np.abs(b), 1e-30)
                err = (np.abs(a.astype(np.float64) - b).max(axis=-1) if a.ndim > 1 else np.abs(a.astype(np.float64) - b)) / scale
                if err.max() <= 1e-6 and bad.mean() < 1e-3:
                    continue
            ok = False
            msg.append(f"{f}: {int(bad.sum())} differ, first at {i}: got {a[i]} want {b[i]} (sx,sy,sz = {ref['sx'][i]},{ref['sy'][i]},{ref['sz'][i]})")
    if not ok:
        raise AssertionError("; ".join(msg))


def check_against_oracle(tag, tm, cloud, origin):
    """Full parity bar on the gathered map (rank 0)."""
    from oracle import oracle as O
    p = default_params(0.2, 0.1, 0.08, origin=origin, origin_is_first_point=0)
    o32, o64 = O.oracle_build(cloud, p, "faithful32"), O.oracle_build(cloud, p, "truth64")
    rep = parity.compare_gathered(tm.gathered_numpy("voxels"), tm.gathered_numpy("columns"), tm.gathered_numpy("slopes"), o32, o64, p)
    assert rep["ok"], f"{tag}: " + json.dumps(rep, default=str)
    print(f"{tag}: parity ok, label mismatches {rep['label_mismatch']} reach mismatches {rep['reach_mismatch']} (all threshold-adjacent)", flush=True)


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    cloud = synthetic.cfg2(1_500_000, scale=0.4)
    origin = [float(v) for v in cloud[0, :3]]
    dev_cloud = torch.from_numpy(cloud).cuda()
    ref_v, ref_s, ref_c = untiled(dev_cloud, origin)

    results = {}
    # NCCL point-to-point, then the library's own exchange with the records pushed by an SM kernel ("sm")
    # and carried by the copy engines ("ce", the default)
    for name, exchange, transport in (("nccl", "nccl", None), ("native-sm", "native", "sm"), ("native", "native", "ce")):
        tm = TiledTwoDmap(0.2, 0.1, 0.08, rank, world, device=local, exchange=exchange, transport=transport, capacity=2_000_000)
        cuts = tm.plan(dev_cloud, origin=origin)
        assert cuts[0] == -32768 and cuts[-1] == 32768 and np.all(np.diff(cuts) >= 0)
        g = tm.build(dev_cloud, "slope", origin=origin, cuts=cuts, filter_points=True)
        got = tm.gathered_numpy()
        sizes = np.diff(g[1].astype(np.int64))
        same_table(f"{name}: gathered voxels vs untiled build", got, ref_v)
        if exchange == "native":
            same_table(f"{name}: gathered slopes vs untiled build", tm.gathered_numpy("slopes"), ref_s)
            same_table(f"{name}: gathered columns vs untiled build", tm.gathered_numpy("columns"), ref_c)
            if rank == 0:
                check_against_oracle("strips " + name, tm, cloud, origin)
                assert sizes.min() > 0.5 * sizes.mean(), f"strips unbalanced: {sizes}"
        results[name] = (tm, cuts, got)
        if rank == 0:
            print(f"multi-gpu {name} ok: strips", sizes.tolist(), flush=True)
    # the two transports must deliver the same bytes
    for which in ("voxels", "slopes", "columns"):
        assert results["native"][0].gathered_numpy(which).tobytes() == results["native-sm"][0].gathered_numpy(which).tobytes(), which
    tm, cuts, got = results["native"]

    # empty strips (ADVICE: equal cuts used to mean "filter off"): rank 0 gets nothing; with >= 3 ranks
    # an empty strip sits BETWEEN two occupied ones, whose boundary rows must still see each other
    if world == 2:
        cuts_e = np.array([-32768, -32768, 32768], np.int32)
    else:
        cuts_e = np.array(cuts, np.int32)
        cuts_e[2] = cuts_e[1]  # strip 1 empty, strip 0 and 2 touch
    tm.build(dev_cloud, "slope", origin=origin, cuts=cuts_e, filter_points=True)
    same_table("empty strip: gathered voxels vs untiled build", tm.gathered_numpy(), ref_v)
    same_table("empty strip: gathered columns vs untiled build", tm.gathered_numpy("columns"), ref_c)
    if rank == 0:
        print("multi-gpu empty-strip ok:", tm.strip_counts[:, 0].tolist(), flush=True)
    if world >= 3:  # the NCCL halo must pair strips 0 and 2 across the empty strip 1 as well
        tn = results["nccl"][0]
        tn.build(dev_cloud, "slope", origin=origin, cuts=cuts_e, filter_points=True)
        same_table("empty strip, nccl: gathered voxels vs untiled build", tn.gathered_numpy(), ref_v)
        if rank == 0:
            print("multi-gpu empty-strip nccl ok:", tn.strip_counts[:, 0].tolist(), flush=True)

    # two builds in flight (depth 2: the gather of the first overlaps the build of the second)
    # must give the same bytes as one-at-a-time builds
    cloud_b = synthetic.cfg2(900_000, scale=0.3)
    dev_b = torch.from_numpy(cloud_b).cuda()
    origin_b = [float(v) for v in cloud_b[0, :3]]
    cuts_b = tm.plan(dev_b, origin=origin_b)
    tm.build(dev_b, "slope", origin=origin_b, cuts=cuts_b, filter_points=True)
    got_b = tm.gathered_numpy().copy()
    pipelined = []
    for transport in ("ce", "sm"):
        tm2 = TiledTwoDmap(0.2, 0.1, 0.08, rank, world, device=local, depth=2, capacity=2_000_000, transport=transport)
        pipelined.append(tm2)
        for rep in range(2):
            tm2.submit(dev_cloud, "slope", origin=origin, cuts=cuts, filter_points=True)
            tm2.submit(dev_b, "slope", origin=origin_b, cuts=cuts_b, filter_points=True)
            ta, _ = tm2.collect()
            ta = ta.cpu().numpy().tobytes()
            tb, _ = tm2.collect()
            tb = tb.cpu().numpy().tobytes()
            assert ta == got.tobytes(), f"pipelined build A differs ({transport}, rep {rep})"  # same strips, same tiles: bytes
            assert tb == got_b.tobytes(), f"pipelined build B differs ({transport}, rep {rep})"
    if rank == 0:
        print("multi-gpu pipelined ok", flush=True)

    # streaming on N GPUs (cfg 4): build from the first 70 % of the cloud, fuse two more scans
    # (every rank is handed the same scan and keeps its strip's points), gather: equals the
    # batch build over the concatenation, to the full parity bar
    na, nb = int(0.7 * len(cloud)), int(0.85 * len(cloud))
    tm3 = TiledTwoDmap(0.2, 0.1, 0.08, rank, world, device=local, capacity=2_000_000)
    tm3.build(dev_cloud[:na].contiguous(), "slope", origin=origin, cuts=cuts, filter_points=True)
    tm3.update(dev_cloud[na:nb].contiguous())
    tm3.update(dev_cloud[nb:].contiguous())
    got_s = tm3.gathered_numpy()
    for f in ("sx", "sy", "sz", "count", "first_index", "column", "slope"):
        assert np.array_equal(got_s[f], ref_v[f]), f"streamed strips: {f}"
    if rank == 0:
        check_against_oracle("streamed strips", tm3, cloud, origin)
    tm3.close()
    dist.barrier()
    for t in [r[0] for r in results.values()] + pipelined:
        t.close()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
