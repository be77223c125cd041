"""The whole per-scan path on the CPU ORACLE ALONE, from raw points (test infrastructure; see gm_oracle.cpp).

Call order = cloud_cb (/root/reference/src/geometric_mapping.cpp:48-125): chopCloud -> getNormals (+ NaN compaction)
-> rvizNormals (VoxelGrid + 1-NN) -> getLocalFrame, then the builder-defined stages (RANSAC plane + cylinder, refit,
labels, polyline).  Every stage is fed the ORACLE's previous output, never the GPU's: comparing `front`/`back`
against the CUDA path verifies the chain end to end (tests/test_gpu_chain.py, bench.py's `parity` object).
"""
from __future__ import annotations

import numpy as np

from . import oracle as O


def front(pts, bound=5.0, radius=0.05, leaf=0.1, wf=0.2, nthreads=0, knn=0, with_nn=True, knn_max_radius=0.0):
    """crop -> normals -> compaction -> VoxelGrid -> 1-NN -> local frame.  knn > 0: k-nearest-neighbour normals."""
    cropped, src = O.crop(pts, bound, True)
    if knn > 0:
        nrm, cnt = O.normals_knn(cropped, knn, cell=max(radius, 1e-3), nthreads=nthreads, max_radius=knn_max_radius)
    else:
        nrm, cnt, _ = O.normals(cropped, radius, mode=0, order=0, nthreads=nthreads)
    cloud, nrm_c, vmap = O.compact(cropped, nrm)
    vox = O.voxel(cloud, leaf)
    nn = None
    if with_nn and vox["V"] > 0:
        # kdtree->nearestKSearch over the PRE-compaction cloud (quirk B.3); the query is the fixed-point centroid
        # the CUDA path defines (within 1e-6 m of PCL's float sum)
        nn, _ = O.nn1_grid(vox["centroids_fx"], cropped, max(radius, 1e-3) * 1.001, nthreads=nthreads)
    fr = O.local_frame(nrm_c, wf)
    return {"cropped": cropped, "crop_src": src, "normals": nrm, "nbr_count": cnt, "cloud": cloud, "normals_c": nrm_c,
            "valid_map": vmap, "vox": vox, "nn_index": nn, "frame": fr, "n_cropped": len(cropped), "n_valid": len(cloud)}


def back(f, ps, cs, tau=0.05, rmin=0.5, rmax=10.0, refit_iters=5, wf=0.2, slice_len=1.0, max_slices=256, nthreads=0):
    """RANSAC plane (ps: H x 3) + cylinder (cs: H x 2) on the oracle's compacted cloud/normals, refit, labels, polyline."""
    cloud, nrm = f["cloud"], f["normals_c"]
    out = {}
    plane = cyl = None
    if ps is not None and len(ps):
        coef, valid = O.plane_hypotheses(cloud, ps)
        counts = O.count_plane(cloud, coef, valid, tau, nthreads=nthreads)
        counts = np.where(valid != 0, counts, -1).astype(np.int32)
        b = O.argmax(counts)
        out.update(plane_coef=coef, plane_valid=valid, plane_counts=counts, plane_best=b)
        if b >= 0:
            plane, prc = O.refit_plane(cloud, coef[b], tau)
            out.update(plane_refit=plane, plane_refit_count=prc)
    if cs is not None and len(cs):
        m7, t12, cvalid = O.cyl_hypotheses(cloud, nrm, cs, rmin, rmax, tau)
        counts = O.count_cyl(cloud, t12, cvalid, nthreads=nthreads)
        counts = np.where(cvalid != 0, counts, -1).astype(np.int32)
        b = O.argmax(counts)
        out.update(cyl_model=m7, cyl_test=t12, cyl_valid=cvalid, cyl_counts=counts, cyl_best=b)
        if b >= 0:
            cyl, crc, crms = O.refit_cylinder(cloud, m7[b], t12[b], refit_iters)
            out.update(cyl_refit=cyl, cyl_refit_count=crc, cyl_refit_rms=crms)
    lab = O.labels(cloud, plane, tau, None if cyl is None else O.cyl_test_params(cyl, tau)[0])
    poly, t0 = O.polyline(cloud, nrm, lab, 2, f["frame"]["vecs"][:, 0], wf, slice_len, max_slices)
    out.update(labels=lab, polyline=poly, polyline_t0=t0)
    return out


# ---------------------------------------------------------------------------------------------------------
# Comparison of a CUDA-path result set with the oracle-alone chain.  `g` = dict of what the C-ABI returned for the
# same raw points and sample indices (tests/test_gpu_chain.py:gpu_chain builds it).  Integer / index / bit-pattern
# outputs are asserted exactly; floating-point outputs are measured and returned (the caller asserts the bars).
def _bits(a):
    """Bit patterns with every NaN mapped to one canonical pattern (the NaN payload is not part of the contract:
    the oracle writes 0x7FC00000, CUDA's CUDART_NAN_F is 0x7FFFFFFF)."""
    b = np.ascontiguousarray(a, np.float32).view(np.uint32).copy()
    b[np.isnan(np.ascontiguousarray(a, np.float32))] = 0x7FC00000
    return b


def gpu_chain(pts, ps, cs, canonical, radius, leaf, bound=5.0, tau=0.05, slice_len=1.0, refit_iters=5, knn=0, knn_max_radius=0.0):
    """The same path on the CUDA library through the C-ABI: everything compare() looks at, downloaded."""
    with gpu_context(len(pts), ps, cs, radius, leaf, bound, tau, slice_len, refit_iters) as ctx:
        ctx.set_normals_mode(1 if canonical else 0)
        if knn:
            ctx.set_knn(knn, max_radius=knn_max_radius)
        ctx.upload_scan(pts)
        ctx.process_scan(ps, cs)
        return gpu_outputs(ctx, ps, cs)


def gpu_context(n, ps, cs, radius, leaf, bound=5.0, tau=0.05, slice_len=1.0, refit_iters=5):
    """A context with the parameters gpu_chain uses, sized for n points and the hypotheses ps / cs."""
    from geometric_mapping_b200 import capi

    H = max(len(ps) if ps is not None else 0, len(cs) if cs is not None else 0, 1)
    prm = capi.default_params(boxFilterBound=bound, neighborRadius=radius, voxelGridLeafSize=leaf, ransacThreshold=tau,
                              sliceLength=slice_len, refitIterations=refit_iters)
    return capi.Context(prm, max_points=max(n, 1), max_hypotheses=H)


def gpu_outputs(ctx, ps, cs):
    """Everything compare() looks at, downloaded from a context after process_scan(ps, cs)."""
    from geometric_mapping_b200 import capi

    c = ctx.counts()
    assert c.device_error == 0
    keys, assign, _ = ctx.download_voxel_assignment()
    vox = ctx.download_voxels()
    g = {"n_cropped": c.n_cropped, "n_valid": c.n_valid, "n_voxels": c.n_voxels, "cropped": ctx.download_cloud(0),
         "normals": ctx.download_normals(0), "nbr_count": ctx.download_neighbor_counts(), "valid_map": ctx.download_valid_map(),
         "cloud": ctx.download_cloud(1), "normals_c": ctx.download_normals(1), "grid6": ctx.voxel_grid(), "vox_key_pt": keys,
         "vox_assign": assign, "vox_keys": vox["keys"], "vox_counts": vox["counts"], "centroids": vox["centroids"],
         "nn_index": vox["nn_index"], "frame": ctx.frame(), "labels": ctx.download_labels(), "polyline": ctx.download_polyline()}
    if ps is not None and len(ps):
        g["plane_coef"], _, g["plane_counts"] = ctx.download_hypotheses(capi.GM_MODEL_PLANE, len(ps))
        g["plane"] = ctx.model(capi.GM_MODEL_PLANE)
    if cs is not None and len(cs):
        g["cyl_model"], g["cyl_test"], g["cyl_counts"] = ctx.download_hypotheses(capi.GM_MODEL_CYLINDER, len(cs))
        g["cyl"] = ctx.model(capi.GM_MODEL_CYLINDER)
    return g


def _angle(a, b):
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    a = a / np.linalg.norm(a, axis=-1, keepdims=True)
    b = b / np.linalg.norm(b, axis=-1, keepdims=True)
    return np.arccos(np.clip(np.abs((a * b).sum(-1)), -1.0, 1.0))


def compare(g, f, b, exact_normals: bool):
    """-> dict of measured divergences.  Raises AssertionError on any exact-contract violation."""
    m = {}
    # ---- exact in every mode: nothing here depends on the float sums of the normals -------------------------
    assert g["n_cropped"] == f["n_cropped"], "n_cropped"
    assert np.array_equal(_bits(g["cropped"]), _bits(f["cropped"])), "cropped cloud"
    assert np.array_equal(g["nbr_count"], f["nbr_count"]), "neighbour counts"
    assert np.array_equal(g["valid_map"], f["valid_map"]), "valid map"
    assert g["n_valid"] == f["n_valid"], "n_valid"
    assert np.array_equal(_bits(g["cloud"]), _bits(f["cloud"])), "compacted cloud"
    v = f["vox"]
    assert g["n_voxels"] == v["V"], "V"
    assert np.array_equal(g["grid6"], v["grid6"]), "voxel lattice"
    assert np.array_equal(g["vox_key_pt"], v["keys"]), "voxel keys"
    assert np.array_equal(g["vox_assign"], v["assign"]), "voxel assignment"
    assert np.array_equal(g["vox_keys"], v["voxel_keys"]) and np.array_equal(g["vox_counts"], v["voxel_counts"]), "voxels"
    assert np.array_equal(_bits(g["centroids"]), _bits(v["centroids_fx"])), "centroids (fixed-point definition)"
    m["centroid_vs_pcl_float_sum_max_m"] = float(np.abs(g["centroids"][:, :3].astype(np.float64) - v["centroids"][:, :3]).max()) if v["V"] else 0.0
    if f["nn_index"] is not None:
        assert np.array_equal(g["nn_index"], f["nn_index"]), "1-NN index"
    if "plane_counts" in b:
        assert np.array_equal(_bits(g["plane_coef"]), _bits(b["plane_coef"])), "plane hypothesis coefficients"
        assert np.array_equal(g["plane_counts"], b["plane_counts"]), "plane inlier counts"
        assert g["plane"]["best_id"] == b["plane_best"], "plane argmax"
    # ---- normals: bit-identical in canonical mode, measured otherwise ----------------------------------------
    gn, on = g["normals"], f["normals"]
    fin = np.isfinite(on[:, 0])
    assert np.array_equal(fin, np.isfinite(gn[:, 0])), "NaN pattern of the normals"
    ang = _angle(gn[fin, :3], on[fin, :3]) if fin.any() else np.zeros(1)
    m["normal_angle_rad"] = {"p50": float(np.percentile(ang, 50)), "p99": float(np.percentile(ang, 99)), "max": float(ang.max())}
    m["curvature_abs_diff_max"] = float(np.abs(gn[fin, 4].astype(np.float64) - on[fin, 4]).max()) if fin.any() else 0.0
    m["normals_bit_identical"] = bool(np.array_equal(_bits(gn), _bits(on)))
    if exact_normals:
        assert m["normals_bit_identical"], "normals (canonical summation order)"
        assert np.array_equal(_bits(g["normals_c"]), _bits(f["normals_c"])), "compacted normals"
    # ---- local frame (tolerance: the 3x3 reduction order is unspecified in Eigen too) --------------------------
    # The oracle accumulates S twice from the same float products w_i*n_i: in float, sequentially (the literal
    # restatement; its own rounding error grows with n: ~5e-4 relative at 1M normals) and in double ("truth").
    fr, orf = g["frame"], f["frame"]
    St = orf["scatter_truth"]
    sn = float(np.abs(St).max())
    tv, tw = np.linalg.eigh(St)
    m["scatter_rel_diff_vs_double"] = float(np.abs(fr["scatter"].astype(np.float64) - St).max() / sn)
    m["eigenvalue_rel_diff_vs_double"] = float(np.abs(fr["vals"].astype(np.float64) - tv).max() / np.abs(tv).max())
    m["axis_angle_rad_vs_double"] = float(_angle(fr["vecs"][:, 0], tw[:, 0]))
    m["scatter_rel_diff"] = float(np.abs(fr["scatter"].astype(np.float64) - orf["scatter"]).max() / sn)
    m["eigenvalue_rel_diff"] = float(np.abs(fr["vals"].astype(np.float64) - orf["vals"]).max() / np.abs(orf["vals"]).max())
    m["axis_angle_rad"] = float(_angle(fr["vecs"][:, 0], orf["vecs"][:, 0]))
    m["float_oracle_scatter_rel_err_vs_double"] = float(np.abs(orf["scatter"].astype(np.float64) - St).max() / sn)
    # ---- cylinder RANSAC: depends on the normals -----------------------------------------------------------
    if "cyl_counts" in b:
        if exact_normals:
            assert np.array_equal(_bits(g["cyl_model"]), _bits(b["cyl_model"])), "cylinder hypothesis coefficients"
            assert np.array_equal(_bits(g["cyl_test"]), _bits(b["cyl_test"])), "cylinder test parameters"
            assert np.array_equal(g["cyl_counts"], b["cyl_counts"]), "cylinder inlier counts"
            assert g["cyl"]["best_id"] == b["cyl_best"], "cylinder argmax"
        both = (g["cyl_counts"] >= 0) & (b["cyl_counts"] >= 0)
        m["cyl_valid_pattern_equal"] = bool(np.array_equal(g["cyl_counts"] >= 0, b["cyl_counts"] >= 0))
        dc = np.abs(g["cyl_counts"][both].astype(np.int64) - b["cyl_counts"][both])
        m["cyl_count_abs_diff"] = {"max": int(dc.max()) if dc.size else 0, "mean": float(dc.mean()) if dc.size else 0.0,
                                   "n_different": int((dc > 0).sum()), "n": int(both.sum())}
        m["cyl_best_id_equal"] = bool(g["cyl"]["best_id"] == b["cyl_best"])
        if b["cyl_best"] >= 0:
            m["cyl_best_count_rel_diff"] = abs(g["cyl"]["best_count"] - int(b["cyl_counts"][b["cyl_best"]])) / max(int(b["cyl_counts"][b["cyl_best"]]), 1)
    # ---- refits (1e-4 relative, north_star) -----------------------------------------------------------------
    if "plane_refit" in b:
        gp, op = g["plane"]["coef"][:4].astype(np.float64), b["plane_refit"].astype(np.float64)
        m["plane_refit_normal_angle_rad"] = float(_angle(gp[:3], op[:3]))
        m["plane_refit_d_abs_diff"] = float(abs(gp[3] - op[3]))
        m["plane_refit_count_equal"] = bool(g["plane"]["refit_count"] == b["plane_refit_count"])
    if "cyl_refit" in b:
        gc, oc = g["cyl"]["coef"][:7].astype(np.float64), b["cyl_refit"].astype(np.float64)
        m["cyl_refit_axis_angle_rad"] = float(_angle(gc[3:6], oc[3:6]))
        m["cyl_refit_radius_rel_diff"] = float(abs(gc[6] - oc[6]) / oc[6])
        d = gc[:3] - oc[:3]
        ax = oc[3:6] / np.linalg.norm(oc[3:6])
        m["cyl_refit_axis_offset_rel"] = float(np.linalg.norm(d - ax * (d @ ax)) / oc[6])  # distance of the GPU's axis point to the oracle's axis / r
        m["cyl_refit_count_rel_diff"] = abs(g["cyl"]["refit_count"] - b["cyl_refit_count"]) / max(b["cyl_refit_count"], 1)
    # ---- labels / polyline -------------------------------------------------------------------------------------
    m["label_mismatch_fraction"] = float((g["labels"] != b["labels"]).mean()) if len(b["labels"]) else 0.0
    gp, op = g["polyline"], b["polyline"]
    m["polyline_slices"] = [int(len(gp)), int(len(op))]
    if len(gp) == len(op) and len(op):
        big = op[:, 7] >= 50
        m["polyline_center_abs_diff_max_m"] = float(np.abs(gp["center"][big].astype(np.float64) - op[big, 0:3]).max()) if big.any() else 0.0
        m["polyline_radius_rel_diff_max"] = float((np.abs(gp["radius"][big] - op[big, 6]) / op[big, 6]).max()) if big.any() else 0.0
        m["polyline_count_abs_diff_max"] = int(np.abs(gp["count"].astype(np.int64) - op[:, 7].astype(np.int64)).max())
    return m
