"""Parity checker: GPU tables (libgndt.so through the C ABI) vs the CPU oracle.

The bar (BASELINE.json north_star):
  * cell assignment, per-cell point counts, layer indices, first-seen order: BIT-EXACT
  * means, scatters, eigenvalues: within REL_TOL = 1e-5, norm-wise (relative to the voxel's
    largest scatter entry / eigenvalue; means relative to max(1, |mean|)), against the
    faithful32 oracle; an excess is accepted only when the GPU value is at least as close to
    the truth64 oracle as faithful32 itself is (the reference's own binary32 noise, H3)
  * labels identical; every mismatch must sit within 1e-5 (relative) of one of the
    thresholds slope_interval / 30 deg / 0.15 m / 100 / the rough==0 test / acos' domain
    edge, and is counted.
"""
import numpy as np

from grid_ndt_b200 import _abi

REL_TOL = 1e-5
LABEL_BITS = _abi.F_FITTED | _abi.F_SLOPE | _abi.F_UP | _abi.F_DOWN
REACH_BITS = _abi.F_REACH_ALL


def _contig(s):
    return np.where(s > 0, s - 1, s)


def compare(gpu_vox, gpu_cols, gpu_slopes, gpu_counts, o32, o64, params, check_reach=True):
    """Returns a report dict; report['ok'] is the verdict.  o32/o64 are oracle.OracleMap."""
    rep = {"ok": True, "fail": []}

    def fail(msg):
        rep["ok"] = False
        rep["fail"].append(msg)

    ov = o32.voxels
    rep["n_voxels"] = (len(gpu_vox), len(ov))
    for k in ("n_binned", "n_dropped", "n_outside_tile", "n_columns", "n_voxels", "n_fitted", "n_slopes"):
        if gpu_counts[k] != o32.counts[k]:
            fail(f"count {k}: gpu {gpu_counts[k]} != oracle {o32.counts[k]}")
    if len(gpu_vox) != len(ov):
        fail("voxel table length differs")
        return rep

    # ---- bit-exact integer fields
    for f in ("sx", "sy", "sz", "count", "first_index"):
        bad = int((gpu_vox[f] != ov[f]).sum())
        rep[f"exact_{f}_mismatch"] = bad
        if bad:
            i = int(np.nonzero(gpu_vox[f] != ov[f])[0][0])
            fail(f"{f}: {bad} mismatches, first at {i}: gpu {gpu_vox[f][i]} oracle {ov[f][i]}")
    if rep["fail"]:
        return rep
    if len(gpu_cols) != len(o32.columns):
        fail("column table length differs")
    else:
        for f in ("sx", "sy", "first_index", "voxel_begin", "voxel_count", "slope_begin", "slope_count"):
            bad = int((gpu_cols[f] != o32.columns[f]).sum())
            if bad and f not in ("slope_begin", "slope_count"):
                fail(f"column {f}: {bad} mismatches")
            rep[f"col_{f}_mismatch"] = bad
        if not np.array_equal(gpu_vox["column"], ov["column"]):
            fail("voxel.column index differs")
        # morton_list order: columns sorted by first_index must reproduce the oracle's list
        order = np.argsort(gpu_cols["first_index"], kind="stable")
        if not np.array_equal(order.astype(np.uint32), o32.morton_list):
            fail("morton_list (first-seen column order) differs")

    fit = (ov["flags"] & _abi.F_FITTED) != 0
    gfit = (gpu_vox["flags"] & _abi.F_FITTED) != 0
    if not np.array_equal(fit, gfit):
        fail("FITTED flag differs")
        return rep
    t64 = o64.voxels

    # ---- means
    g, a, t = gpu_vox["mean"][fit].astype(np.float64), ov["mean"][fit].astype(np.float64), t64["mean"][fit].astype(np.float64)
    scale = np.maximum(1.0, np.abs(a).max(axis=1, keepdims=True))
    err = np.abs(g - a) / scale
    exc = err.max(axis=1) > REL_TOL
    explained = np.abs(g - t).max(axis=1) <= np.abs(a - t).max(axis=1) + 1e-7 * scale[:, 0]
    rep["mean_max_rel_err"] = float(err.max()) if err.size else 0.0
    rep["mean_excess"] = int(exc.sum())
    rep["mean_excess_unexplained"] = int((exc & ~explained).sum())
    if rep["mean_excess_unexplained"]:
        fail(f"mean: {rep['mean_excess_unexplained']} voxels beyond 1e-5 and not explained by truth64")
    rep["mean_max_rel_err_vs_truth64"] = float((np.abs(g - t) / scale).max()) if err.size else 0.0
    unf = ~fit
    if np.abs(gpu_vox["mean"][unf]).max(initial=0) != 0 or np.abs(gpu_vox["scatter"][unf]).max(initial=0) != 0:
        fail("unfitted voxels must keep the constructor's zero centroid/scatter")

    # ---- scatter
    g, a, t = gpu_vox["scatter"][fit].astype(np.float64), ov["scatter"][fit].astype(np.float64), t64["scatter"][fit].astype(np.float64)
    snorm = np.maximum(np.abs(t).max(axis=1), 1e-30)
    err = np.abs(g - a).max(axis=1) / snorm
    exc = err > REL_TOL
    explained = np.abs(g - t).max(axis=1) <= np.abs(a - t).max(axis=1) + 1e-6 * snorm
    rep["scatter_max_rel_err"] = float(err.max()) if err.size else 0.0
    rep["scatter_excess"] = int(exc.sum())
    rep["scatter_excess_unexplained"] = int((exc & ~explained).sum())
    rep["scatter_max_rel_err_vs_truth64"] = float((np.abs(g - t).max(axis=1) / snorm).max()) if err.size else 0.0
    if rep["scatter_excess_unexplained"]:
        fail(f"scatter: {rep['scatter_excess_unexplained']} voxels beyond 1e-5 and not explained by truth64")

    # ---- eigenvalues (relative to lambda_max), rough, normals
    g, a, t = gpu_vox["evals"][fit].astype(np.float64), ov["evals"][fit].astype(np.float64), t64["evals"][fit].astype(np.float64)
    lmax = np.maximum(np.abs(t).max(axis=1), 1e-30)
    err = np.abs(g - a).max(axis=1) / lmax
    exc = err > REL_TOL
    explained = np.abs(g - t).max(axis=1) <= np.abs(a - t).max(axis=1) + 1e-6 * lmax
    rep["evals_max_rel_err"] = float(err.max()) if err.size else 0.0
    rep["evals_excess"] = int(exc.sum())
    rep["evals_excess_unexplained"] = int((exc & ~explained).sum())
    rep["evals_max_rel_err_vs_truth64"] = float((np.abs(g - t).max(axis=1) / lmax).max()) if err.size else 0.0
    if rep["evals_excess_unexplained"]:
        fail(f"evals: {rep['evals_excess_unexplained']} voxels beyond 1e-5 and not explained by truth64")

    gr, ar = gpu_vox["rough"][fit].astype(np.float64), ov["rough"][fit].astype(np.float64)
    rerr = np.abs(gr - ar) / lmax
    rbad = rerr > REL_TOL
    # the rough==0 -> 0.01 rule (map2D.h:131): a mismatch is threshold-adjacent when the
    # oracle's smallest eigenvalue is within 1e-5*lambda_max of zero
    zero_adj = rbad & (np.abs(a[:, 0]) <= REL_TOL * lmax) & ((gr == np.float32(0.01)) | (ar == np.float32(0.01)))
    rough_expl = rbad & ~zero_adj & (np.abs(g[:, 0] - t[:, 0]) <= np.abs(a[:, 0] - t[:, 0]) + 1e-6 * lmax)
    rep["rough_mismatch"] = int(rbad.sum())
    rep["rough_zero_rule_adjacent"] = int(zero_adj.sum())
    rep["rough_unexplained"] = int((rbad & ~zero_adj & ~rough_expl).sum())
    if rep["rough_unexplained"]:
        fail(f"rough: {rep['rough_unexplained']} unexplained mismatches")

    gn, an = gpu_vox["normal"][fit].astype(np.float64), ov["normal"][fit].astype(np.float64)
    gn /= np.maximum(np.linalg.norm(gn, axis=1, keepdims=True), 1e-30)
    an /= np.maximum(np.linalg.norm(an, axis=1, keepdims=True), 1e-30)
    ang = np.arccos(np.clip(np.abs((gn * an).sum(axis=1)), 0.0, 1.0))
    gap = (t[:, 1] - t[:, 0]) / lmax
    well = gap > 1e-3
    allow = 1e-4 + 4e-5 / np.maximum(gap, 1e-12)
    nbad = well & (ang > allow)
    # the same rule as for the scatters (H3): far from the origin faithful32's own binary32 noise tilts ITS
    # normal; a difference is accepted when the GPU normal is at least as close to truth64's as faithful32's is
    tn = t64["normal"][fit].astype(np.float64)
    tn /= np.maximum(np.linalg.norm(tn, axis=1, keepdims=True), 1e-30)
    ang_gt = np.arccos(np.clip(np.abs((gn * tn).sum(axis=1)), 0.0, 1.0))
    ang_at = np.arccos(np.clip(np.abs((an * tn).sum(axis=1)), 0.0, 1.0))
    nexpl = nbad & (ang_gt <= ang_at + 1e-6)
    rep["normal_checked"] = int(well.sum())
    rep["normal_max_angle_rad"] = float(ang[well].max()) if well.any() else 0.0
    rep["normal_max_angle_rad_vs_truth64"] = float(ang_gt[well].max()) if well.any() else 0.0
    rep["normal_excess"] = int(nbad.sum())
    rep["normal_mismatch"] = int((nbad & ~nexpl).sum())
    if rep["normal_mismatch"]:
        fail(f"normal: {rep['normal_mismatch']} well-conditioned normals differ and are not explained by truth64")
    unit = np.abs(np.linalg.norm(gpu_vox["normal"][fit].astype(np.float64), axis=1) - 1.0)
    if unit.size and unit.max() > 1e-5:
        fail("normals are not unit length")

    # ---- labels: up / down / slope
    gl, al = gpu_vox["flags"] & LABEL_BITS, ov["flags"] & LABEL_BITS
    lbad_all = np.nonzero(gl != al)[0]
    rep["label_mismatch"] = int(lbad_all.size)
    # a mismatch where the GPU agrees with the truth64 oracle is the reference's own
    # binary32 noise (H3), counted separately; the rest must be threshold-adjacent
    agree64 = (gpu_vox["flags"] & LABEL_BITS)[lbad_all] == (t64["flags"] & LABEL_BITS)[lbad_all]
    rep["label_mismatch_agreeing_with_truth64"] = int(agree64.sum())
    lbad = lbad_all[~agree64]
    interval = float(params.slope_interval)
    n_adj = 0
    cz = _contig(ov["sz"])
    for i in lbad:
        # recompute the oracle's |dz| against both vertical neighbours; adjacent if either
        # sits within 1e-5 (relative) of slope_interval
        adj = False
        for j in (i - 1, i + 1):
            if 0 <= j < len(ov) and ov["sx"][j] == ov["sx"][i] and ov["sy"][j] == ov["sy"][i] and abs(int(cz[j]) - int(cz[i])) == 1:
                for zj in (float(ov["mean"][j][2]), 0.0):
                    dz = abs(zj - float(ov["mean"][i][2]))
                    if abs(dz - interval) <= REL_TOL * max(dz, interval):
                        adj = True
        n_adj += adj
    rep["label_mismatch_threshold_adjacent"] = n_adj
    if lbad.size != n_adj:
        fail(f"labels: {lbad.size - n_adj} up/down/slope mismatches are NOT threshold-adjacent")

    # ---- reach bits (only meaningful when labels agree on the Slope set)
    if check_reach:
        gr_, ar_ = gpu_vox["flags"] & REACH_BITS, ov["flags"] & REACH_BITS
        rb_all = np.nonzero(gr_ != ar_)[0]
        rep["reach_mismatch"] = int(rb_all.size)
        agree64 = gr_[rb_all] == (t64["flags"] & REACH_BITS)[rb_all]
        rep["reach_mismatch_agreeing_with_truth64"] = int(agree64.sum())
        rb = rb_all[~agree64]
        rep["reach_mismatch_threshold_adjacent"] = _reach_adjacent(rb, ov, o32.columns, params) if rb.size else 0
        if rb.size != rep["reach_mismatch_threshold_adjacent"]:
            fail(f"reach bits: {rb.size - rep['reach_mismatch_threshold_adjacent']} mismatches are NOT threshold-adjacent")

    # column slope_begin / slope_count follow from the labels: with identical labels they must be identical
    if rep["label_mismatch"] == 0 and (rep.get("col_slope_begin_mismatch", 0) or rep.get("col_slope_count_mismatch", 0)):
        fail(f"column slope_begin/slope_count differ ({rep['col_slope_begin_mismatch']}/{rep['col_slope_count_mismatch']}) although all labels agree")

    # ---- slope table consistency with the voxel table
    is_slope = (gpu_vox["flags"] & _abi.F_SLOPE) != 0
    if len(gpu_slopes) != int(is_slope.sum()):
        fail("slope table length != number of SLOPE voxels")
    else:
        idx = np.nonzero(is_slope)[0]
        if not (np.array_equal(gpu_slopes["voxel"], idx.astype(np.uint32)) and np.array_equal(gpu_slopes["sz"], gpu_vox["sz"][idx])
                and np.array_equal(gpu_slopes["mean"], gpu_vox["mean"][idx]) and np.array_equal(gpu_slopes["normal"], gpu_vox["normal"][idx])
                and np.array_equal(gpu_slopes["rough"], gpu_vox["rough"][idx]) and np.array_equal(gpu_slopes["flags"], gpu_vox["flags"][idx])):
            fail("slope table does not mirror the voxel table")
    return rep


def compare_gathered(vox, cols, slopes, o32, o64, params, check_reach=True):
    """The same bar for a map assembled from several GPUs' strips: counts are derived from the
    gathered tables themselves (no strip may have lost or duplicated a record)."""
    counts = {"n_binned": int(vox["count"].sum()), "n_dropped": o32.counts["n_dropped"], "n_outside_tile": 0,
              "n_columns": len(cols), "n_voxels": len(vox), "n_fitted": int(((vox["flags"] & _abi.F_FITTED) != 0).sum()),
              "n_slopes": len(slopes)}
    return compare(vox, cols, slopes, counts, o32, o64, params, check_reach=check_reach)


def assemble_strips(strips):
    """Host statement of what the device-side push (csrc/gndt_exchange.cuh, xchg_push_kernel) does
    to strip-local indices: strips = [(voxels, columns)] in rank order -> (voxels, columns) of the
    whole map.  voxel.column += columns before, voxel.slope += slopes before (unless none),
    column.voxel_begin += voxels before, column.slope_begin += slopes before."""
    vox_off = col_off = slope_off = 0
    vs, cs = [], []
    for v, c in strips:
        v, c = v.copy(), c.copy()
        v["column"] += np.uint32(col_off)
        has = v["slope"] != 0xFFFFFFFF
        v["slope"][has] += np.uint32(slope_off)
        c["voxel_begin"] += np.uint32(vox_off)
        c["slope_begin"] += np.uint32(slope_off)
        vox_off, col_off, slope_off = vox_off + len(v), col_off + len(c), slope_off + int(has.sum())
        vs.append(v)
        cs.append(c)
    return np.concatenate(vs), np.concatenate(cs)


def _angle(n1, n2):
    d = float(np.dot(n1, n2)) / (float(np.linalg.norm(n1)) * float(np.linalg.norm(n2)) + 1e-300)
    a = np.degrees(np.arccos(np.clip(d, -1, 1)))
    return 180 - a if a > 90 else a, d


def _reach_adjacent(idx, ov, cols, params):
    """How many reach-bit mismatches have a candidate edge within 1e-5 of a threshold."""
    key = {(int(c["sx"]), int(c["sy"])): c for c in cols}
    nxt = lambda s: 1 if s == -1 else s + 1
    prv = lambda s: -1 if s == 1 else s - 1
    n_adj = 0
    for i in idx:
        v = ov[i]
        adj = False
        sx, sy = int(v["sx"]), int(v["sy"])
        for nb in ((sx, prv(sy)), (sx, nxt(sy)), (nxt(sx), sy), (prv(sx), sy)):
            c = key.get(nb)
            if c is None:
                continue
            for j in range(int(c["voxel_begin"]), int(c["voxel_begin"] + c["voxel_count"])):
                u = ov[j]
                if not (u["flags"] & _abi.F_SLOPE):
                    continue
                ang, d = _angle(u["normal"].astype(np.float64), v["normal"].astype(np.float64))
                dz = abs(float(u["mean"][2]) - float(v["mean"][2]))
                if (abs(ang - params.angle_max_deg) <= REL_TOL * params.angle_max_deg or abs(dz - params.reach_height) <= REL_TOL * params.reach_height
                        or abs(float(u["rough"]) - params.rough_max) <= REL_TOL * params.rough_max or abs(abs(d) - 1.0) <= 1e-6):
                    adj = True
        n_adj += adj
    return n_adj


def run_case(cloud, params, demand="slope", device=None, check_reach=True):
    """Build on the GPU through the TwoDmap mirror and compare with both oracle modes."""
    from grid_ndt_b200 import TwoDmap
    from oracle import oracle as O

    params.demand = _abi.GNDT_DEMAND_SLOPE if demand == "slope" else _abi.GNDT_DEMAND_TRUE
    m = TwoDmap(params.grid_len, params.z_len, device=device)
    m.setInterval(params.slope_interval)
    m.params.min_points = params.min_points
    m.params.normalize_cov = params.normalize_cov
    m.params.rough_max, m.params.angle_max_deg, m.params.reach_height = params.rough_max, params.angle_max_deg, params.reach_height
    m.params.tile_lo, m.params.tile_hi = params.tile_lo, params.tile_hi
    if params.origin_is_first_point:
        m.chatterCallback(cloud, demand)
    else:
        m.setCloudFirst([params.origin[i] for i in range(3)])
        m.uniformDivision(cloud)
        m.create2DMap(demand)
    counts = m.counts()
    host_cloud = cloud.cpu().numpy() if hasattr(cloud, "cpu") else cloud
    o32 = O.oracle_build(host_cloud, params, "faithful32")
    o64 = O.oracle_build(host_cloud, params, "truth64")
    rep = compare(m.voxels, m.columns, m.slopes, counts, o32, o64, params, check_reach=check_reach)
    rep["stage_ms"] = m.stage_ms()
    rep["counts"] = counts
    m.close()
    return rep


if __name__ == "__main__":  # debug CLI: python -m tests.parity cfg1 [n]
    import json
    import sys

    from grid_ndt_b200 import synthetic
    from grid_ndt_b200._abi import default_params

    name = sys.argv[1] if len(sys.argv) > 1 else "cfg1"
    n = int(sys.argv[2]) if len(sys.argv) > 2 else 200_000
    if name == "bridge":
        from oracle import oracle as O
        cloud, _ = O.bridge_ground()
        p = default_params(0.1, 0.05, 0.08)
    else:
        spec = synthetic.CONFIGS[name]
        kw = {"scale": (n / spec.n) ** 0.5} if name == "cfg2" else ({"extent": 224.0 * (n / spec.n) ** 0.5} if name == "cfg3" else {})
        cloud = synthetic.make(name, n, **kw)
        p = default_params(spec.grid_len, spec.z_len, spec.slope_interval)
    rep = run_case(cloud, p)
    print(json.dumps(rep, indent=1, default=str))
    sys.exit(0 if rep["ok"] else 1)
