"""TwoDmap::AccessibleNeighbors (map2D.h:530-548) over a (slopes, columns) table pair, in numpy.

The exact rule the traversability graph (csrc/gndt_graph.cuh) and the reach bits (edges_kernel,
csrc/gndt_label.cuh) are held to.  It works on any table pair: a GPU map's own tables, a gathered
multi-GPU map, an oracle build (oracle_tables) or tables made by hand.

Neighbour cells are the contiguous (cx, cy) +- 1 cells in the order left (cy - 1), right (cy + 1),
forward (cx + 1), back (cx - 1), found by np.searchsorted on the sorted column keys; inside a cell
the Slopes keep slope-table order.  The predicate is `reachable` / `count_angle` in the kernel's own
mixed precision, which numpy reproduces step for step:
  * binary32 dot product, one rounding per multiply and per add;
  * binary64 norms (sum of squares in binary64, correctly rounded sqrt);
  * res = binary64 quotient dot / (l1 * l2), stored to binary32;
  * deg = acos(res) * 180 in binary32, / pi in binary64, stored to binary32; folded to 180 - deg above 90;
  * fabsf(tz - mz) <= reach_height in binary32, rough <= rough_max, no F_UP on the target.
The one step that is not exactly reproducible is acosf, documented by CUDA to within 2 ulp.  The
reference takes the correctly rounded binary32 arccos and evaluates the angle test for it and for
every float up to ACOS_ULP ulp on either side.  A candidate edge is decided (True or False) when
all of them agree and UNDECIDED otherwise; only undecided edges may differ from the kernels.
"""
from dataclasses import dataclass

import numpy as np

from grid_ndt_b200 import _abi
from grid_ndt_b200._abi import COLUMN_DTYPE, SLOPE_DTYPE

ACOS_ULP = 2
TRUE, FALSE, UNDECIDED = 1, 0, -1
REACH = (_abi.F_REACH_L, _abi.F_REACH_R, _abi.F_REACH_F, _abi.F_REACH_B)
DIRS = ((0, -1), (0, 1), (1, 0), (-1, 0))  # (dx, dy) of left, right, forward, back


def contig(s):
    """Contiguous index of a signed index (no gap at the -1/+1 crossing)."""
    s = np.asarray(s, np.int64)
    return np.where(s > 0, s - 1, s)


def signed(c):
    """Signed index of a contiguous index."""
    c = np.asarray(c, np.int64)
    return np.where(c >= 0, c + 1, c)


def _key(cx, cy):
    return (np.asarray(cx, np.int64) + 32768) * 65536 + (np.asarray(cy, np.int64) + 32768)


def f32(x):
    return np.asarray(x, np.float32)


def normal_length(n):
    """normal_length: binary64 squares and sums in the kernel's order, then sqrt."""
    n = np.asarray(n, np.float32).astype(np.float64)
    return np.sqrt((n[..., 0] * n[..., 0] + n[..., 1] * n[..., 1]) + n[..., 2] * n[..., 2])


def angle_res(a, b):
    """count_angle's res: (float)((double)dot32(a, b) / (l1 * l2))."""
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    dot = a[..., 0] * b[..., 0]
    dot = dot + a[..., 1] * b[..., 1]
    dot = dot + a[..., 2] * b[..., 2]
    with np.errstate(divide="ignore", invalid="ignore"):
        return (dot.astype(np.float64) / (normal_length(a) * normal_length(b))).astype(np.float32)


def angle_from_acos(ac):
    """count_angle after acosf: degrees via *180 (binary32) and /pi (binary64), folded to <= 90."""
    deg = f32(ac) * np.float32(180.0)
    an = (deg.astype(np.float64) / np.pi).astype(np.float32)
    return np.where(an > np.float32(90.0), np.float32(180.0) - an, an)


def acos_candidates(res):
    """(k, ...) binary32 values acosf may return for res: the correctly rounded value and every
    float up to ACOS_ULP ulp on either side of it."""
    with np.errstate(invalid="ignore"):
        c = np.arccos(np.asarray(res, np.float32).astype(np.float64)).astype(np.float32)
    out, lo, hi = [c], c, c
    for _ in range(ACOS_ULP):
        lo, hi = np.nextafter(lo, np.float32(-np.inf)), np.nextafter(hi, np.float32(np.inf))
        out += [lo, hi]
    return np.stack(out)


def angle_verdict(res, angle_max_deg):
    """TRUE / FALSE / UNDECIDED for count_angle(...) <= angle_max_deg, given res."""
    with np.errstate(invalid="ignore"):
        ok = angle_from_acos(acos_candidates(res)) <= np.float32(angle_max_deg)
    return np.where(ok.all(axis=0), TRUE, np.where(ok.any(axis=0), UNDECIDED, FALSE)).astype(np.int8)


def other_tests(t_rough, t_z, t_flags, mz, params):
    """countReachable's tests other than the angle: no F_UP, rough <= rough_max, |tz - mz| <= reach_height."""
    dz = np.abs(f32(t_z) - f32(mz))
    return (((np.asarray(t_flags, np.uint32) & _abi.F_UP) == 0) & (f32(t_rough) <= np.float32(params.rough_max))
            & (dz <= np.float32(params.reach_height)))


def verdict(t, s, params):
    """Verdict of 'Slope record t is reachable from Slope record s' (arrays broadcast)."""
    base = other_tests(t["rough"], t["mean"][..., 2], t["flags"], s["mean"][..., 2], params)
    ang = angle_verdict(angle_res(t["normal"], s["normal"]), params.angle_max_deg)
    return np.where(base, ang, FALSE).astype(np.int8)


def columns_of(slopes):
    """The column table of a slope table sorted by (cx, cy): one column per cell that holds a Slope
    (cells without one contribute no candidate, so the graph and the reach bits do not change)."""
    key = _key(contig(slopes["sx"]), contig(slopes["sy"]))
    if len(key) and np.any(np.diff(key) < 0):
        raise ValueError("slope table not sorted by (cx, cy)")
    first = np.nonzero(np.r_[True, np.diff(key) != 0])[0] if len(key) else np.zeros(0, np.int64)
    cols = np.zeros(len(first), COLUMN_DTYPE)
    cols["sx"], cols["sy"] = slopes["sx"][first], slopes["sy"][first]
    cols["slope_begin"] = first
    cols["slope_count"] = np.diff(np.r_[first, len(slopes)])
    return cols


@dataclass
class Graph:
    """Every candidate edge of every Slope, in the kernels' visiting order (L, R, F, B cell, slope
    order inside a cell): candidates of Slope i are [cand_off[i], cand_off[i + 1])."""
    cand_off: np.ndarray   # int64 [S + 1]
    cand_src: np.ndarray   # int64, source Slope of each candidate
    cand_tgt: np.ndarray   # int64, target Slope
    cand_dir: np.ndarray   # int8, 0..3 = L, R, F, B
    verdict: np.ndarray    # int8, TRUE / FALSE / UNDECIDED
    nb: np.ndarray         # int64 [S, 4]: column of each neighbour cell, -1 for none

    @property
    def n_undecided(self):
        return int((self.verdict == UNDECIDED).sum())

    def csr(self):
        """(offsets, targets) of the decided-True edges."""
        sel = self.verdict == TRUE
        deg = np.bincount(self.cand_src[sel], minlength=len(self.cand_off) - 1)
        return np.r_[0, np.cumsum(deg)].astype(np.uint32), self.cand_tgt[sel].astype(np.uint32)


def neighbour_columns(slopes, columns):
    """[S, 4] column index of the left, right, forward and back cell of every Slope, -1 for none."""
    S, C = len(slopes), len(columns)
    nb = np.full((S, 4), -1, np.int64)
    if not S or not C:
        return nb
    keys = _key(contig(columns["sx"]), contig(columns["sy"]))
    if np.any(np.diff(keys) <= 0):
        raise ValueError("column table not sorted strictly by (cx, cy)")
    cx, cy = contig(slopes["sx"]), contig(slopes["sy"])
    for d, (dx, dy) in enumerate(DIRS):
        want = _key(cx + dx, cy + dy)
        j = np.minimum(np.searchsorted(keys, want), C - 1)
        nb[:, d] = np.where(keys[j] == want, j, -1)
    return nb


def graph_reference(slopes, columns, params):
    """The candidate edges of every Slope of the table pair with their verdicts (a Graph)."""
    slopes = np.asarray(slopes, SLOPE_DTYPE)
    columns = np.asarray(columns, COLUMN_DTYPE)
    S = len(slopes)
    nb = neighbour_columns(slopes, columns)
    begin = np.where(nb >= 0, columns["slope_begin"][np.maximum(nb, 0)].astype(np.int64) if len(columns) else 0, 0)
    count = np.where(nb >= 0, columns["slope_count"][np.maximum(nb, 0)].astype(np.int64) if len(columns) else 0, 0)
    cnt = count.reshape(-1)
    total = int(cnt.sum())
    starts = np.r_[0, np.cumsum(cnt)[:-1]] if len(cnt) else np.zeros(0, np.int64)
    within = np.arange(total, dtype=np.int64) - np.repeat(starts, cnt)
    tgt = np.repeat(begin.reshape(-1), cnt) + within
    src = np.repeat(np.repeat(np.arange(S, dtype=np.int64), 4), cnt)
    dirs = np.repeat(np.tile(np.arange(4, dtype=np.int8), S), cnt)
    off = np.r_[0, np.cumsum(count.sum(axis=1))].astype(np.int64)
    v = verdict(slopes[tgt], slopes[src], params) if total else np.zeros(0, np.int8)
    return Graph(off, src, tgt, dirs, v, nb)


def rows(off, tgt):
    """The CSR (off, tgt) as one tuple of targets per Slope."""
    return [tuple(tgt[off[i]:off[i + 1]]) for i in range(len(off) - 1)]


def graph_errors(off, tgt, ref):
    """Why the CSR (off, tgt) breaks the exact rule against a Graph, or [] when it follows it:
    every list is a subsequence of its Slope's candidates (order kept, no repeats) that holds
    every decided-True candidate and no decided-False one."""
    off, tgt = np.asarray(off, np.int64), np.asarray(tgt, np.int64)
    S = len(ref.cand_off) - 1
    if len(off) != S + 1:
        return [f"offsets has {len(off)} entries, not n_slopes + 1 = {S + 1}"]
    if off[0] != 0 or np.any(np.diff(off) < 0) or off[-1] != len(tgt):
        return ["offsets are not a CSR index of the targets"]
    errs = []
    src = np.repeat(np.arange(S, dtype=np.int64), np.diff(off))
    ckey = ref.cand_src * (S + 1) + ref.cand_tgt  # candidates are unique per Slope
    order = np.argsort(ckey, kind="stable")
    gkey = src * (S + 1) + tgt
    j = np.minimum(np.searchsorted(ckey[order], gkey), max(len(ckey) - 1, 0))
    found = (len(ckey) > 0) & (tgt >= 0) & (tgt < S)
    found = found & (ckey[order][j] == gkey) if len(ckey) else np.zeros(len(tgt), bool)
    if not found.all():
        i = int(np.nonzero(~found)[0][0])
        errs.append(f"{int((~found).sum())} targets are not candidates (first: Slope {src[i]} -> {tgt[i]})")
        return errs
    pos = order[j]
    same = src[1:] == src[:-1]
    if np.any(same & (np.diff(pos) <= 0)):
        i = int(src[1:][same & (np.diff(pos) <= 0)][0])
        errs.append(f"the list of Slope {i} is out of the reference's order or repeats a target")
    bad_false = ref.verdict[pos] == FALSE
    if bad_false.any():
        i = int(np.nonzero(bad_false)[0][0])
        errs.append(f"{int(bad_false.sum())} decided-unreachable targets listed (first: Slope {src[i]} -> {tgt[i]})")
    present = np.zeros(len(ref.verdict), bool)
    present[pos] = True
    missing = (ref.verdict == TRUE) & ~present
    if missing.any():
        i = int(np.nonzero(missing)[0][0])
        errs.append(f"{int(missing.sum())} decided-reachable targets missing (first: Slope {ref.cand_src[i]} -> {ref.cand_tgt[i]})")
    return errs


def assert_graph(off, tgt, slopes, columns, params, label=""):
    """The CSR equals AccessibleNeighbors of the tables exactly, up to undecided edges; returns the
    reference Graph and prints its undecided-edge count."""
    ref = graph_reference(slopes, columns, params)
    errs = graph_errors(off, tgt, ref)
    print(f"\n{label}graph: {len(slopes)} Slopes, {len(tgt)} edges, {ref.n_undecided} undecided candidate edges")
    assert not errs, "; ".join(errs)
    return ref


def reach_bit_errors(slopes, params, columns=None):
    """(errors, undecided directions) of the slopes' GNDT_F_REACH_* bits against the exact rule: a
    direction with a decided-True candidate has its bit set, one whose candidates are all
    decided-False (or that has none) has it clear."""
    slopes = np.asarray(slopes, SLOPE_DTYPE)
    ref = graph_reference(slopes, columns_of(slopes) if columns is None else columns, params)
    S = len(slopes)
    idx = ref.cand_src * 4 + ref.cand_dir
    any_true = np.zeros(S * 4, bool)
    any_und = np.zeros(S * 4, bool)
    any_true[idx[ref.verdict == TRUE]] = True
    any_und[idx[ref.verdict == UNDECIDED]] = True
    bits = (np.asarray(slopes["flags"], np.uint32)[:, None] & np.array(REACH, np.uint32)[None, :]) != 0
    bits = bits.reshape(-1)
    must_set = any_true & ~bits
    must_clear = ~any_true & ~any_und & bits
    errs = []
    for what, sel in (("set", must_set), ("clear", must_clear)):
        if sel.any():
            i = int(np.nonzero(sel)[0][0])
            errs.append(f"{int(sel.sum())} reach bits should be {what} (first: Slope {i // 4}, direction {'LRFB'[i % 4]})")
    return errs, int((any_und & ~any_true).sum())


def assert_reach_bits(slopes, params, columns=None, label=""):
    errs, und = reach_bit_errors(slopes, params, columns)
    print(f"\n{label}reach bits: {len(slopes)} Slopes, {und} undecided directions")
    assert not errs, "; ".join(errs)


def oracle_tables(o):
    """(slopes, columns) of an oracle build: the SLOPE voxels in table order, and its columns."""
    v = o.voxels
    sl = v[(v["flags"] & _abi.F_SLOPE) != 0]
    s = np.zeros(len(sl), SLOPE_DTYPE)
    for f in ("sx", "sy", "sz", "mean", "normal", "rough", "flags"):
        s[f] = sl[f]
    s["voxel"] = np.nonzero((v["flags"] & _abi.F_SLOPE) != 0)[0]
    return s, o.columns.copy()
