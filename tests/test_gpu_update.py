"""Streaming fusion (gndt_update / TwoDmap.change2DMap) — BASELINE configs[3].

The reference's incremental path is dead code with an inconsistent formula (SURVEY Q13), so
the contract is batch equivalence: a map built from cloud A and updated with scans B1..Bk
equals one build over the concatenation A+B1+..+Bk, with the same parity bar as a build."""
import numpy as np
import pytest

from grid_ndt_b200 import _abi, synthetic
from grid_ndt_b200._abi import default_params

pytestmark = pytest.mark.gpu


def _gpu():
    import torch
    if not torch.cuda.is_available():
        pytest.fail("gpu-marked test on a box without CUDA (no fallback exists)")
    return torch


def _check_against_batch(m, cloud, p):
    from oracle import oracle as O
    from tests import parity
    o32 = O.oracle_build(cloud, p, "faithful32")
    o64 = O.oracle_build(cloud, p, "truth64")
    rep = parity.compare(m.voxels, m.columns, m.slopes, m.counts(), o32, o64, p)
    assert rep["ok"], rep["fail"]
    return rep


@pytest.mark.parametrize("demand", ["slope", "true"])
def test_update_equals_batch_build(demand):
    _gpu()
    from grid_ndt_b200 import TwoDmap
    cloud = synthetic.cfg2(900_000, scale=0.3)
    cuts = [0, 400_000, 520_000, 521_000, 760_000, 900_000]
    m = TwoDmap(0.2, 0.1)
    m.setInterval(0.08)
    m.chatterCallback(cloud[: cuts[1]], demand)
    for a, b in zip(cuts[1:-1], cuts[2:]):
        m.change2DMap(cloud[a:b])
    p = default_params(0.2, 0.1, 0.08, demand)
    rep = _check_against_batch(m, cloud, p)
    assert rep["counts"] if "counts" in rep else True
    assert m.counts()["n_input"] == 900_000 and m.counts()["n_binned"] == 899_999
    m.close()


def test_update_grows_capacity_and_accepts_device_scans():
    torch = _gpu()
    from grid_ndt_b200 import TwoDmap
    cloud = synthetic.cfg3(600_000, extent=40.0)
    m = TwoDmap(0.1, 0.1)
    m.setInterval(0.08)
    m.chatterCallback(cloud[:20_000], "slope")  # tiny resident map, then 29x more voxels arrive
    v0 = m.counts()["n_voxels"]
    m.change2DMap(torch.from_numpy(cloud[20_000:300_000]).cuda())
    m.change2DMap(cloud[300_000:])
    assert m.counts()["n_voxels"] > 5 * v0
    _check_against_batch(m, cloud, default_params(0.1, 0.1, 0.08))
    m.close()


def test_scans_from_cfg4_generator():
    """BASELINE configs[3] shape: lidar discs fused into the cfg2 scene at high rate."""
    _gpu()
    from grid_ndt_b200 import TwoDmap
    base = synthetic.cfg2(400_000, scale=0.2)
    scans = list(synthetic.scans(6, 20_000, radius=4.0, cfg2_scale=0.2))
    m = TwoDmap(0.2, 0.1)
    m.setInterval(0.08)
    m.chatterCallback(base, "slope")
    for s in scans:
        m.change2DMap(s)
        ms = m.stage_ms()
        assert ms["total"] < 50.0
    _check_against_batch(m, np.concatenate([base] + scans), default_params(0.2, 0.1, 0.08))
    m.close()


def test_update_requires_a_resident_map():
    _gpu()
    from grid_ndt_b200 import GndtError, TwoDmap
    m = TwoDmap(0.2, 0.1)
    with pytest.raises(GndtError) as e:
        m.change2DMap(np.zeros((10, 4), np.float32))  # map2D.h:679: change2DMap on an empty map fails
    assert e.value.status == _abi.GNDT_ERR_STATE
    m.close()


def test_cell_center_and_origin():
    _gpu()
    from grid_ndt_b200 import TwoDmap
    cloud = synthetic.cfg1(50_000)
    m = TwoDmap(0.2, 0.1)
    m.chatterCallback(cloud, "slope")
    assert np.array_equal(m.origin(), cloud[0, :3])
    v = m.voxels
    fit = np.nonzero(v["flags"] & 1)[0][:2000]
    for i in fit[::97]:
        c = m.countPositionXYZ(int(v["sx"][i]), int(v["sy"][i]), int(v["sz"][i]))
        assert np.all(np.abs(c - v["mean"][i]) <= np.array([0.1, 0.1, 0.05]) + 1e-4)  # mean lies inside its cell
        key, z = m.transMortonXYZ(c)
        assert z == int(v["sz"][i])
    m.close()


def _touched_columns(scan, origin, gl):
    """The reference's changeMorton_list for one scan (src/receiver.cpp:47-56): the (sx, sy) of the
    scan's points in first-touched order, with the x-y index arithmetic of map2D.h:950-972 in binary32."""
    def idx(v, o):
        d = (np.abs(v - np.float32(o)) / np.float32(gl)).astype(np.float32)
        n = np.maximum(np.ceil(d), 1).astype(np.int64)
        return np.where(v > np.float32(o), n, -n)
    sx, sy = idx(scan[:, 0], origin[0]), idx(scan[:, 1], origin[1])
    seen, out = set(), []
    for k in zip(sx.tolist(), sy.tolist()):
        if k not in seen:
            seen.add(k)
            out.append(k)
    return out


def test_changed_columns_is_the_references_change_list():
    _gpu()
    from grid_ndt_b200 import TwoDmap
    base = synthetic.cfg2(400_000, scale=0.2)
    scans = list(synthetic.scans(3, 20_000, radius=4.0, cfg2_scale=0.2))
    m = TwoDmap(0.2, 0.1)
    m.setInterval(0.08)
    m.chatterCallback(base, "slope")
    for s in scans:
        m.change2DMap(s)
        cols = m.columns
        got = [(int(c["sx"]), int(c["sy"])) for c in cols[m.changed_columns]]
        want = _touched_columns(s, base[0, :3], 0.2)
        assert got == want, (len(got), len(want))
        assert m.changeMorton_list[0] == m.transMortonXYZ(s[0, :3])[0]
    m.close()


def test_remove_undoes_update():
    """build(A) + update(B) + remove(B) == build(A): §8(f)4 (del2DMap, map2D.h:826-915)."""
    _gpu()
    from grid_ndt_b200 import TwoDmap
    cloud = synthetic.cfg2(700_000, scale=0.25)
    a, b = cloud[:450_000], cloud[450_000:]
    m = TwoDmap(0.2, 0.1)
    m.setInterval(0.08)
    m.chatterCallback(a, "slope")
    ref_v, ref_c = m.voxels.copy(), m.columns.copy()
    m.change2DMap(b)
    assert m.counts()["n_voxels"] > len(ref_v)
    m.del2DMap(b)
    v, c = m.voxels, m.columns
    assert len(v) == len(ref_v) and len(c) == len(ref_c)
    for f in ("sx", "sy", "sz", "count", "first_index", "column", "slope"):
        assert np.array_equal(v[f], ref_v[f]), f
    assert m.counts()["n_input"] == 450_000 and m.counts()["n_binned"] == 449_999
    # the full parity bar against the oracle's build of A alone (floats differ from the GPU's own
    # build of A only by the rounding of the merge and its inverse)
    _check_against_batch(m, a, default_params(0.2, 0.1, 0.08))
    touched = {(int(x["sx"]), int(x["sy"])) for x in c[m.changed_columns]}
    want = set(_touched_columns(b, a[0, :3], 0.2)) & {(int(x["sx"]), int(x["sy"])) for x in c}
    assert touched == want  # cells that vanished with the scan are not listed
    m.close()


def test_failed_update_and_remove_leave_the_map_unchanged():
    """ADVICE r1: a capacity overflow used to leave the resident map half-fused.  The halo rows
    of the map are checked too: a failed call must not change what gndt_halo_pack sends."""
    torch = _gpu()
    from grid_ndt_b200 import GndtError, TwoDmap, lib
    from grid_ndt_b200.builder import _check
    cap = 65536

    def halo():  # first and last x row of m, packed into fresh zeroed buffers
        bufs = torch.zeros(2, (cap + 1) * _abi.VOXEL_DTYPE.itemsize, dtype=torch.uint8, device="cuda")
        _check(m._h, lib().gndt_halo_pack(m._h, bufs[0].data_ptr(), bufs[1].data_ptr(), cap, 0))
        torch.cuda.synchronize()
        return bufs.cpu().numpy().tobytes()

    cloud = synthetic.cfg2(500_000, scale=0.22)
    a, b = cloud[:300_000], cloud[300_000:]
    m = TwoDmap(0.2, 0.1)
    m.setInterval(0.08)
    m.chatterCallback(a, "slope")
    n0 = m.counts()["n_voxels"]
    m.close()
    m = TwoDmap(0.2, 0.1)
    m.setInterval(0.08)
    m.params.max_voxels = n0 + 10  # room for the map of A, not for A + B
    m.chatterCallback(a, "slope")
    before = (m.voxels.tobytes(), m.slopes.tobytes(), m.columns.tobytes(), m.counts())
    halo_before = halo()
    hdr = np.frombuffer(halo_before, np.uint32).reshape(2, -1)[:, :3]  # count, cx, overflow of each row
    assert (hdr[:, 0] > 0).all() and (hdr[:, 2] == 0).all() and hdr[0, 0] + hdr[1, 0] < before[3]["n_voxels"]
    m.change2DMap(b)
    with pytest.raises(GndtError) as e:
        m.counts()
    assert e.value.status == _abi.GNDT_ERR_CAPACITY
    assert (m.voxels.tobytes(), m.slopes.tobytes(), m.columns.tobytes(), m.counts()) == before
    assert halo() == halo_before
    m.del2DMap(b)  # never fused
    with pytest.raises(GndtError) as e:
        m.counts()
    assert e.value.status == _abi.GNDT_ERR_STATE
    assert (m.voxels.tobytes(), m.slopes.tobytes(), m.columns.tobytes(), m.counts()) == before
    assert halo() == halo_before
    m.params.max_voxels = 0
    # changing the cell size under a resident map is refused (two key spaces cannot be fused)
    m.setLen(0.3)
    import ctypes as C
    from grid_ndt_b200 import lib
    lib().gndt_set_params(m._h, C.byref(m.params))
    with pytest.raises(GndtError):
        m.change2DMap(b)
    m.close()
