"""Multi-GPU map build: one x strip of the map per GPU of a single box, one process per GPU.

Default exchange ("native"): the halo rows and the gather of the finished tables go through
peer-mapped memory inside libgndt.so (gndt_xchg_*, csrc/gndt_exchange.cuh): no NCCL kernel, no
host synchronisation for the strip sizes, strip-local indices made global while the records are
pushed.  torch.distributed only carries the 128-byte buffer handles between the ranks once, at
construction.  The older NCCL point-to-point form (exchange="nccl") is kept for comparison and
is what the rest of this docstring describes.

Everything up to and including the surface labels depends only on the points of one x-y
column (SURVEY.md §8(e)), so strips need no exchange while they are built.  The only cross-
strip dependence is the forward/back reachability of the first and last x row of a strip, so
those two rows (a thin halo, fixed-size buffers, no host round trip) are swapped with the two
neighbour strips BEFORE the gather and each rank finishes its own boundary rows.  Then the
strip sizes are all-gathered (the only host synchronisation of a build) and every rank sends
its final records straight out of the builder's table into the other ranks' copy of the whole
map (batched point-to-point = an all-gather with uneven sizes, no padding, no staging copies;
measured faster than padded all_gather / broadcasts, tools/gather_bench.py).  Last, strip-local
column / slope indices are made global by adding per-strip offsets.

Back-to-back builds (`depth` > 1): the gather is NVLink work and the build is SM work, so
`submit()` / `collect()` rotate through `depth` independent builders (handle, stream, halo and
map buffers each) and the record gather of cloud i runs while cloud i+1 is being built.  The
halo + size exchange and the record gather use two NCCL communicators so that neither queues
behind the other.  torch.distributed is only the plumbing (process groups, streams, buffers).
"""
import ctypes as C
from collections import deque
from typing import Optional

import numpy as np
import torch
import torch.distributed as dist

from . import _abi
from ._abi import COLUMN_DTYPE, SLOPE_DTYPE, VOXEL_DTYPE, XchgInfo, XchgView
from ._lib import lib
from .builder import TwoDmap, _check

REC = VOXEL_DTYPE.itemsize  # 96


class _Slot:
    """One builder with everything a build in flight owns."""

    def __init__(self, res, zres, interval, world, device, halo_records, own_stream):
        self.map = TwoDmap(res, zres, device=device)
        self.map.setInterval(interval)
        self.device = torch.device("cuda", self.map._device)
        self.stream = torch.cuda.Stream(self.device) if own_stream else None
        self.counts = torch.zeros(world * 4, dtype=torch.int32, device=self.device)
        self.halo = torch.zeros(4 * (halo_records + 1) * REC, dtype=torch.uint8, device=self.device) if halo_records else None
        self.table = None
        self.g_slopes = self.g_columns = None
        self.offsets = None
        self.strip_counts = None


class Gathered(tuple):
    """Result of collect(): unpacks as (voxel table or None, offsets) like before, and carries the
    gathered slope / column tables and the per-strip counts as attributes."""

    def __new__(cls, table, offsets, **kw):
        obj = super().__new__(cls, (table, offsets))
        obj.__dict__.update(kw)
        return obj


def allgather_bytes(blob: bytes, world: int, group=None, device=None) -> list:
    """Every rank's fixed-size byte blob, in rank order (the one collective of the native
    exchange: buffer handles at construction).  CPU tensors with gloo, CUDA tensors with NCCL."""
    t = torch.frombuffer(bytearray(blob), dtype=torch.uint8)
    if device is not None:
        t = t.to(device)
    out = torch.empty(world * len(blob), dtype=torch.uint8, device=t.device)
    dist.all_gather_into_tensor(out, t, group=group)
    raw = out.cpu().numpy().tobytes()
    return [raw[i * len(blob):(i + 1) * len(blob)] for i in range(world)]


class TiledTwoDmap:
    """Strip r of `world` strips.  `cuts` are contiguous signed x column indices; strip r
    keeps columns with cuts[r] <= cx < cuts[r+1] (gndt_params.tile_lo/hi)."""

    def __init__(self, res, zres, interval, rank: int, world: int, device: Optional[int] = None, group=None,
                 halo_records: int = 32768, depth: int = 1, exchange: str = "native", gather=("voxels", "slopes", "columns"),
                 capacity: int = 8_000_000, transport: Optional[str] = None):
        """exchange: "native" (peer-mapped memory inside libgndt.so) or "nccl" (point-to-point).
        transport (native only): "ce" = the records travel by copy engine (gndt_xchg_stage / gndt_xchg_send: one
        512-byte host round trip per build, hidden behind the builds already queued; does not slow the build
        running beside it), "sm" = pushed by an SM kernel (gndt_xchg_run: no host round trip, but the build
        beside it on the sending GPU slows down by about the duration of the push).  Default: "ce"
        (GNDT_XCHG_TRANSPORT overrides).
        gather: which tables of the whole map every rank ends up with (native only; the planner reads
        slopes + columns).  capacity: voxels of the WHOLE map the gathered tables can hold (native)."""
        self.rank, self.world, self.group = rank, world, group
        self.halo_records = halo_records  # capacity of one halo row (records); overflow is reported, not truncated
        self.exchange = exchange if world > 1 else "nccl"  # one strip: nothing to exchange
        import os
        self.transport = transport or os.environ.get("GNDT_XCHG_TRANSPORT", "ce")
        if self.transport not in ("ce", "sm"):
            raise ValueError(f"transport {self.transport!r}: 'ce' or 'sm'")
        self.what = sum({"voxels": _abi.X_VOXELS, "slopes": _abi.X_SLOPES, "columns": _abi.X_COLUMNS}[g] for g in gather)
        self.slots = [_Slot(res, zres, interval, world, device, halo_records if self.exchange == "nccl" else 0, own_stream=depth > 1)
                      for _ in range(depth)]
        self.gather_group = group
        if self.exchange == "native":
            L = lib()
            infos = b""
            for s in self.slots:
                mine = XchgInfo()
                _check(s.map._h, L.gndt_xchg_create(s.map._h, rank, world, int(capacity), int(halo_records), self.what, C.byref(mine)))
                infos += bytes(mine)
            every = allgather_bytes(infos, world, group, self.slots[0].device if dist.get_backend(group) == "nccl" else None)
            for k, s in enumerate(self.slots):
                arr = (XchgInfo * world)()
                for r in range(world):
                    C.memmove(C.byref(arr[r]), every[r][k * 128:(k + 1) * 128], 128)
                _check(s.map._h, L.gndt_xchg_connect(s.map._h, arr, world))
        elif depth > 1 and world > 1:
            # second communicator: the record gather of build i must not queue behind the halo /
            # size exchange of build i+1 (collective: every rank constructs its TiledTwoDmap)
            self.gather_group = dist.new_group(ranks=list(range(world))) if group is None else dist.new_group(
                ranks=dist.get_process_group_ranks(group))
        self.build_stream = None
        self.map = self.slots[0].map
        self.device = self.slots[0].device
        self._next = 0
        self._inflight = deque()
        self._last = self.slots[0]
        self._cuts = None  # strip boundaries of the resident build (update() keeps them)

    @property
    def depth(self) -> int:
        return len(self.slots)

    @property
    def pending(self) -> int:
        """Builds submitted and not yet collected."""
        return len(self._inflight)

    @property
    def last_map(self) -> TwoDmap:
        """The builder of the build most recently collected (its strip-local tables, counts,
        stage times)."""
        return self._last.map

    @property
    def offsets(self):
        return self._last.offsets

    @property
    def strip_counts(self):
        return self._last.strip_counts

    def plan(self, cloud, origin=None) -> np.ndarray:
        """Balanced cuts from a histogram over x columns.  Every rank that sees the same
        cloud computes the same cuts; no communication."""
        if origin is not None:
            self.map.setCloudFirst(origin)
        return self.map.plan_tiles(cloud, self.world)

    # ---- phase 1: everything that needs no size on the host ---------------------------------
    def submit(self, cloud, demand="slope", origin=None, cuts=None, filter_points=True, update=False):
        """Start a build on the next builder (asynchronous): local strip build (labels are per
        column: no communication), thin halo swapped with the two neighbour strips, own boundary
        rows finished, strip sizes all-gathered on the device.  update=True fuses `cloud` (one
        more scan, the same on every rank: each keeps the points of its strip) into the strip
        map that builder already holds instead of starting a new one (streaming, cfg 4)."""
        if len(self._inflight) == self.depth:
            raise RuntimeError("all builders busy: collect() before submitting another cloud")
        if update and self.depth != 1:
            raise RuntimeError("streaming updates need depth == 1: the resident map lives in one builder")
        s = self.slots[self._next]
        self._next = (self._next + 1) % self.depth
        m, L = s.map, lib()
        if not update:
            if origin is not None:
                m.setCloudFirst(origin)
            self._cuts = np.asarray(cuts, np.int64) if cuts is not None and filter_points else None
            if cuts is not None and filter_points:
                lo, hi = int(cuts[self.rank]), int(cuts[self.rank + 1])
                # an empty strip (equal cuts: one x row holds more than its share of the points)
                # must keep NOTHING; lo >= hi would mean "filter off"
                m.setTile(*((lo, hi) if lo < hi else _abi.TILE_EMPTY))
            else:
                m.setTile(0, 0)
        if self.exchange == "native" and self.depth > 1:
            return self._submit_pipelined(s, cloud, demand)
        stream = s.stream if s.stream is not None else torch.cuda.current_stream(s.device)
        if s.stream is not None:
            s.stream.wait_stream(torch.cuda.current_stream(s.device))  # the cloud was produced there
        with torch.cuda.stream(stream):
            st = stream.cuda_stream
            if update:
                m.change2DMap(cloud, stream=st)
            else:
                m.uniformDivision(cloud)
                m.create2DMap(demand, stream=st)
            if self.exchange == "native":
                # halo rows, strip sizes, gather, index fix-up: all inside the library, all on this stream
                if self.transport == "ce":
                    _check(m._h, L.gndt_xchg_stage(m._h, st))
                    _check(m._h, L.gndt_xchg_send(m._h, st))  # depth 1: nothing else to enqueue meanwhile
                else:
                    _check(m._h, L.gndt_xchg_run(m._h, st))
                s.sent = True
                self._inflight.append(s)
                return s
            slot_b = (self.halo_records + 1) * REC
            send_first, send_last, recv_prev, recv_next = (s.halo[i * slot_b:(i + 1) * slot_b] for i in range(4))
            _check(m._h, L.gndt_halo_pack(m._h, send_first.data_ptr(), send_last.data_ptr(), self.halo_records, st))
            prev, nxt = halo_peers(self._cuts, self.rank, self.world)
            ops = []
            if prev is not None:
                ops += [dist.P2POp(dist.isend, send_first, prev, group=self.group),
                        dist.P2POp(dist.irecv, recv_prev, prev, group=self.group)]
            if nxt is not None:
                ops += [dist.P2POp(dist.isend, send_last, nxt, group=self.group),
                        dist.P2POp(dist.irecv, recv_next, nxt, group=self.group)]
            if ops:
                for req in dist.batch_isend_irecv(ops):
                    req.wait()
            _check(m._h, L.gndt_halo_edges(m._h, recv_prev.data_ptr() if prev is not None else None,
                                           recv_next.data_ptr() if nxt is not None else None, st))
            p_cnt = C.c_void_p()
            _check(m._h, L.gndt_device_count_ptr(m._h, C.byref(p_cnt)))
            mine = _as_tensor(p_cnt.value, 16, s.device).view(torch.int32)
            dist.all_gather_into_tensor(s.counts, mine, group=self.group)
        self._inflight.append(s)
        return s

    def _submit_pipelined(self, s, cloud, demand):
        """depth > 1, native exchange.  Builds run ONE AFTER THE OTHER on a shared build stream (three builds
        time-slicing the SMs would all finish late and their exchanges would then pile up behind them); what
        overlaps is the exchange of build i (this builder's own stream, NVLink-bound, few SMs) with the kernels of
        build i + 1, and the upload of a host cloud (this builder's stream as well) with everything before it."""
        m, L = s.map, lib()
        if self.build_stream is None:
            self.build_stream = torch.cuda.Stream(s.device)
            for t in self.slots:
                t.build_done, t.xchg_done, t.staged = torch.cuda.Event(enable_timing=True), torch.cuda.Event(), torch.cuda.Event()
                t.build_start = torch.cuda.Event(enable_timing=True)
                t.dev_cloud = None
        bs = self.build_stream
        cur = torch.cuda.current_stream(s.device)
        if isinstance(cloud, torch.Tensor) and cloud.is_cuda:
            bs.wait_stream(cur)  # the cloud was produced there
            src = cloud
        else:  # host cloud: upload on the builder's own stream, beside the builds in flight
            host = cloud if isinstance(cloud, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(cloud, dtype=np.float32))
            if s.dev_cloud is None or s.dev_cloud.shape != host.shape:
                s.dev_cloud = torch.empty(host.shape, dtype=torch.float32, device=s.device)
            with torch.cuda.stream(s.stream):
                s.dev_cloud.copy_(host, non_blocking=True)  # ordered behind this builder's previous exchange
                s.staged.record(s.stream)
            bs.wait_event(s.staged)
            src = s.dev_cloud
        bs.wait_event(s.xchg_done)  # this builder's tables and exchange buffer are free again
        with torch.cuda.stream(bs):
            s.build_start.record(bs)
            m.uniformDivision(src)
            m.create2DMap(demand, stream=bs.cuda_stream)
            s.build_done.record(bs)
        s.stream.wait_event(s.build_done)
        if self.transport == "ce":
            _check(m._h, L.gndt_xchg_stage(m._h, s.stream.cuda_stream))
            s.sent = False
            self._inflight.append(s)
            self._send_ready()  # earlier builds whose counts have landed meanwhile
            return s
        with torch.cuda.stream(s.stream):
            _check(m._h, L.gndt_xchg_run(m._h, s.stream.cuda_stream))
            s.xchg_done.record(s.stream)
        s.sent = True
        self._inflight.append(s)
        return s

    def _send(self, s):
        """Copy-engine transport, second half: blocks the host until the strip counts of build `s` are here."""
        if getattr(s, "sent", True):
            return
        _check(s.map._h, lib().gndt_xchg_send(s.map._h, s.stream.cuda_stream))
        s.xchg_done.record(s.stream)
        s.sent = True

    def _send_ready(self):
        """Issue, in order and without blocking, the transfers of the builds in flight whose counts have landed."""
        L = lib()
        for s in self._inflight:
            if getattr(s, "sent", True):
                continue
            rc = L.gndt_xchg_counts_ready(s.map._h)
            _check(s.map._h, min(rc, 0))
            if rc != 1:
                break
            self._send(s)

    def wait_oldest(self):
        """Pipelined native exchange: block until the oldest build in flight has been exchanged; returns its
        builder WITHOUT reading sizes or tables (probes and benchmarks; collect() is the full form)."""
        s = self._inflight.popleft()
        self._send(s)
        s.xchg_done.synchronize()
        self._last = s
        return s

    # ---- phase 2: sizes on the host (the one synchronisation), records to every rank ---------
    def collect(self):
        """Finish the OLDEST build in flight: returns (table tensor [V_total, 96] uint8 on this
        rank's GPU, offsets[world+1]).  The gather and the index fix-up are enqueued on the
        builder's stream; synchronise it (or the device) before reading the table on the host.
        The table is valid until that builder is used again (`depth` submits later)."""
        if not self._inflight:
            raise RuntimeError("nothing submitted")
        s = self._inflight.popleft()
        m, L = s.map, lib()
        stream = s.stream if s.stream is not None else torch.cuda.current_stream(s.device)
        if self.exchange == "native":
            self._send(s)
            self._send_ready()
            v = XchgView()
            _check(m._h, L.gndt_xchg_view_get(m._h, C.byref(v)))  # synchronises this builder's stream only
            w = self.world
            sv = np.array(v.strip_voxels[:w], np.int64)
            s.strip_counts = np.stack([sv, np.array(v.strip_columns[:w], np.int64), np.array(v.strip_slopes[:w], np.int64),
                                       np.zeros(w, np.int64)], 1)
            s.offsets = np.concatenate([[0], np.cumsum(sv)]).astype(np.uint64)
            view = lambda ptr, n, rec: (_as_tensor(ptr, max(int(n), 1) * rec, s.device)[: int(n) * rec].view(-1, rec) if ptr else None)
            s.table = view(v.voxels, v.n_voxels, REC)
            s.g_slopes = view(v.slopes, v.n_slopes, SLOPE_DTYPE.itemsize)
            s.g_columns = view(v.columns, v.n_columns, COLUMN_DTYPE.itemsize)
            self._last = s
            return Gathered(s.table, s.offsets, slopes=s.g_slopes, columns=s.g_columns, strip_counts=s.strip_counts,
                            n_voxels=int(v.n_voxels), n_slopes=int(v.n_slopes), n_columns=int(v.n_columns))
        with torch.cuda.stream(stream):
            st = stream.cuda_stream
            counts4 = s.counts.cpu().numpy().astype(np.int64).reshape(self.world, 4)  # {voxels, columns, slopes, fitted}
            counts = counts4[:, 0]
            s.offsets = np.concatenate([[0], np.cumsum(counts)]).astype(np.uint64)
            col_off = np.concatenate([[0], np.cumsum(counts4[:, 1])])[:-1].astype(np.uint32)
            slope_off = np.concatenate([[0], np.cumsum(counts4[:, 2])])[:-1].astype(np.uint32)
            total, n = int(s.offsets[-1]), int(counts[self.rank])
            if s.table is None or s.table.numel() < max(total, 1) * REC:
                s.table = torch.empty(int(max(total, 1) * 1.25) * REC, dtype=torch.uint8, device=s.device)
            table = s.table
            p_tab, cap = C.c_void_p(), C.c_size_t()
            _check(m._h, L.gndt_device_table_ptr(m._h, C.byref(p_tab), C.byref(cap)))
            local = _as_tensor(p_tab.value, max(n, 1) * REC, s.device)[: n * REC]
            lo = int(s.offsets[self.rank]) * REC
            ops = []
            for r in range(self.world):
                if r == self.rank or counts[r] == 0:
                    continue
                ops.append(dist.P2POp(dist.irecv, table[int(s.offsets[r]) * REC: int(s.offsets[r + 1]) * REC], r,
                                      group=self.gather_group))
            if n:
                for r in range(self.world):
                    if r != self.rank:
                        ops.append(dist.P2POp(dist.isend, local, r, group=self.gather_group))
                table[lo: lo + n * REC].copy_(local, non_blocking=True)
            if ops:
                for req in dist.batch_isend_irecv(ops):
                    req.wait()
            off = (C.c_uint64 * (self.world + 1))(*[int(x) for x in s.offsets])
            co = (C.c_uint32 * self.world)(*[int(x) for x in col_off])
            so = (C.c_uint32 * self.world)(*[int(x) for x in slope_off])
            _check(m._h, L.gndt_apply_strip_offsets(m._h, table.data_ptr(), off, co, so, self.world, st))
        s.strip_counts = counts4
        self._last = s
        return table[: total * REC].view(-1, REC), s.offsets

    def build(self, cloud, demand="slope", origin=None, cuts=None, filter_points=True):
        """One build, start to finish: submit() + collect().  `cloud` may be the whole cloud
        (filter_points=True: points of other strips are dropped on the device) or only this
        strip's share."""
        self.submit(cloud, demand, origin=origin, cuts=cuts, filter_points=filter_points)
        return self.collect()

    def update(self, scan):
        """Fuse one more scan into the strips and re-assemble the whole map on every rank
        (change2DMap on N GPUs: every rank is handed the same scan and keeps its strip's
        points; SURVEY.md §8(e), cfg 4).  Needs a map built with build(..., cuts=...)."""
        self.submit(scan, update=True)
        return self.collect()

    def join(self):
        """Make the current stream wait for everything enqueued on the builders' streams."""
        for s in self._inflight:
            self._send(s)
        cur = torch.cuda.current_stream(self.device)
        if self.build_stream is not None:
            cur.wait_stream(self.build_stream)
        for s in self.slots:
            if s.stream is not None:
                cur.wait_stream(s.stream)

    def synchronize(self):
        for s in self._inflight:
            self._send(s)
        if self.build_stream is not None:
            self.build_stream.synchronize()
        for s in self.slots:
            if s.stream is not None:
                s.stream.synchronize()
        torch.cuda.current_stream(self.device).synchronize()

    def gathered_numpy(self, which: str = "voxels") -> np.ndarray:
        """The gathered voxel (or, native exchange, slope / column) table of the last collected build."""
        self.synchronize()
        s = self._last
        if self.exchange == "native":
            t, dt = {"voxels": (s.table, VOXEL_DTYPE), "slopes": (s.g_slopes, SLOPE_DTYPE), "columns": (s.g_columns, COLUMN_DTYPE)}[which]
            if t is None:
                raise RuntimeError(f"{which} were not gathered (gather=...)")
            return t.cpu().numpy().reshape(-1).view(dt)
        total = int(s.offsets[-1])
        return s.table[: total * REC].cpu().numpy().view(VOXEL_DTYPE).reshape(-1)

    def close(self):
        for s in self.slots:
            s.map.close()


def halo_peers(cuts, rank: int, world: int):
    """(lower, upper) halo peer of `rank`, None at an end of the map: the nearest ranks whose strip
    [cuts[r], cuts[r+1]) is not empty.  An empty strip (equal cuts) keeps nothing and swaps no rows,
    and the strips on either side of it swap theirs with each other, since their x rows may touch.
    Every rank derives the same pairs from the same cuts, so each send has its matching receive.
    cuts = None (no strip filter): the ranks either side."""
    if cuts is None:
        return (rank - 1 if rank > 0 else None), (rank + 1 if rank + 1 < world else None)
    full = [r for r in range(world) if cuts[r] < cuts[r + 1]]
    if rank not in full:
        return None, None
    i = full.index(rank)
    return (full[i - 1] if i > 0 else None), (full[i + 1] if i + 1 < len(full) else None)


def _as_tensor(ptr: int, nbytes: int, device) -> torch.Tensor:
    """Zero-copy uint8 view of library-owned device memory (valid until the next build)."""

    class _Holder:
        pass

    h = _Holder()
    h.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (ptr, False), "version": 3}
    return torch.as_tensor(h, device=device)
