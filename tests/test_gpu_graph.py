"""The traversability graph built on the GPU (gndt_build_edges, csrc/gndt_graph.cuh) on synthetic
clouds, held to the exact rule of tests/graph_reference.py on the GPU's own tables: same lists, same
order, for every Slope, up to edges whose angle test acosf's 2-ulp freedom leaves undecided.  The
reference itself is pinned to the oracle's AccessibleNeighbors in test_gpu_graph_boundaries.py.
The 4 reach bits are exactly "the list has a Slope in that direction"."""
import numpy as np
import pytest

from grid_ndt_b200 import _abi, synthetic
from grid_ndt_b200._abi import default_params

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("name,n,gl,kw,demand", [
    ("cfg1", 300_000, 0.2, {}, "slope"),
    ("cfg2", 600_000, 0.2, {"scale": 0.25}, "slope"),
    ("cfg2", 400_000, 0.2, {"scale": 0.2}, "true"),
    ("cfg3", 400_000, 0.1, {"extent": 20.0}, "slope"),
])
def test_graph_equals_oracle(name, n, gl, kw, demand):
    import torch
    if not torch.cuda.is_available():
        pytest.fail("gpu-marked test on a box without CUDA (no fallback exists)")
    from grid_ndt_b200 import TwoDmap
    from tests import graph_reference as G
    cloud = synthetic.make(name, n, **kw)
    p = default_params(gl, 0.1, 0.08, demand)
    m = TwoDmap(gl, 0.1)
    m.setInterval(0.08)
    m.chatterCallback(cloud, demand)
    off, tgt = m.edges()
    sl, cols = m.slopes, m.columns
    assert len(off) == len(sl) + 1
    G.assert_graph(off, tgt, sl, cols, p, f"{name} {demand}: ")
    # reach bits <=> a target in that direction's cell
    cont = lambda s: np.where(s > 0, s - 1, s)
    cx, cy = cont(sl["sx"]).astype(np.int64), cont(sl["sy"]).astype(np.int64)
    deg = np.diff(off.astype(np.int64))
    src = np.repeat(np.arange(len(sl)), deg)
    dx, dy = cx[tgt] - cx[src], cy[tgt] - cy[src]
    bits = np.zeros(len(sl), np.uint32)
    for mask, sel in ((_abi.F_REACH_L, (dx == 0) & (dy == -1)), (_abi.F_REACH_R, (dx == 0) & (dy == 1)),
                      (_abi.F_REACH_F, (dx == 1) & (dy == 0)), (_abi.F_REACH_B, (dx == -1) & (dy == 0))):
        np.bitwise_or.at(bits, src[sel], np.uint32(mask))
    assert np.all((np.abs(dx) + np.abs(dy)) == 1), "a target outside the 4-neighbourhood"
    assert np.array_equal(bits, sl["flags"] & _abi.F_REACH_ALL), "reach bits disagree with the graph"
    m.close()
