"""Shared input preparation for the parity tests (numpy only; no arithmetic that is under test)."""
import numpy as np

from line3dpp_b200 import synth


def pair_inputs(scene, src, tgt):
    """Float inputs of one view pair exactly as matchingGPU hands them to match_lines_GPU (line3D.cc:1040-1064):
    float RtKinv / C of both views, float F.  No translation (kernel-level tests do not need it)."""
    RtKinv, C = synth.camera_blocks(scene)
    F = synth.fundamental(scene.K[src], scene.R[src], scene.t[src], scene.K[tgt], scene.R[tgt], scene.t[tgt])
    f32 = lambda a: np.ascontiguousarray(a, np.float32)
    return dict(ls=scene.segs[src], lt=scene.segs[tgt], F=f32(F).reshape(9), Rs=f32(RtKinv[src]).reshape(9),
                Rt=f32(RtKinv[tgt]).reshape(9), Cs=f32(C[src]), Ct=f32(C[tgt]))


def scene_descs(scene, k=None):
    """l3d_view_desc[] for a scene (double camera blocks from numpy; float copies made by capi.make_view_descs)."""
    from line3dpp_b200 import capi
    RtKinv, C = synth.camera_blocks(scene)
    V = scene.num_views
    k = np.zeros(V, np.float32) if k is None else k
    return capi.make_view_descs(scene.cam_ids, [scene.width] * V, [scene.height] * V, [len(s) for s in scene.segs],
                                RtKinv, C, C, k, np.zeros(V, np.float32))


def pair_F(scene, pairs):
    out = np.zeros((len(pairs), 9), np.float32)
    for i, (s, t) in enumerate(pairs):
        out[i] = synth.fundamental(scene.K[s], scene.R[s], scene.t[s], scene.K[t], scene.R[t], scene.t[t]).astype(np.float32).reshape(9)
    return out


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


# ---------------------------------------------------------------------------------------------- recorded reference outputs
# The parity tests compare with outputs of the unmodified reference that are stored under tests/golden/ (make_ref_outputs.py).
# Bit-exact comparisons keep a SHA-256 of the canonical bytes; toleranced ones keep a fixed, seeded sample of the values.
IDS = ("src_cam", "src_seg", "tgt_cam", "tgt_seg")
GEO = ("overlap", "d_p1", "d_p2", "d_q1", "d_q2")


def sha(*arrays):
    import hashlib
    h = hashlib.sha256()
    for a in arrays:
        a = np.ascontiguousarray(a)
        h.update(f"{a.dtype.str}{a.shape}".encode())
        h.update(a.tobytes())
    return h.hexdigest()


def pick(n):
    """fixed, seeded sample of at most 64 indices out of n (sorted); depends on n only"""
    return np.sort(np.random.default_rng(0).choice(n, min(n, 256), replace=False))[::4]


def match_sha(m, score=True):
    """ids, overlap, depths (and score3D) of match records, as raw bits"""
    return sha(*[np.asarray(m[f]).astype(np.uint32) for f in IDS], *[bits(m[f]) for f in GEO + (("score3D",) if score else ())])


def list_sha(counts, recs, fields=("tgt_seg", "overlap", "d_p1", "d_p2", "d_q1", "d_q2")):
    """kNN lists in slot order: counts + the first counts[r] records of every row"""
    rows = [recs[r, :counts[r]] for r in range(len(counts))]
    cat = np.concatenate(rows) if rows else recs[:0, 0]
    return sha(np.asarray(counts, np.int64), *[bits(cat[f]) if recs.dtype[f].kind == "f" else cat[f].astype(np.int64) for f in fields])


def row_shas(counts, recs):
    """per row: 32 bits of the digest of its match set (order-free)"""
    return np.array([int(sha(np.array(r, np.int64))[:8], 16) for r in rows_as_sets(counts, recs)], np.uint32)


def tie_sha(counts, recs):
    """the kNN lists up to exact ties at the k-th place: per row the multiset of overlaps and the set of matches whose overlap is
    above the row's smallest one (the reference pops an unordered heap, so which of several equal k-th candidates is kept is
    unspecified)"""
    out = []
    for row in rows_as_sets(counts, recs):
        kth = min((e[1] for e in row), default=-1)
        out.append((sorted(e[1] for e in row), sorted(e for e in row if e[1] != kth)))
    return sha(np.frombuffer(repr(out).encode(), np.uint8))


def sorted_endpoints(s):
    """3D segments with their two end points in a fixed order (the sign of the principal axis is free)"""
    return np.sort(np.stack([s["p1"], s["p2"]], 1), axis=1).reshape(-1, 6)


def stage_record(pairs=None, scored=None, kept=None, view_info=None, estimates=None, collinear=None, l2g=None, aff_raw=None,
                 aff=None, num_lines=None, residuals=None, segments=None, exact_scores=True):
    """canonical record of the stages of a Line3D run; every argument is what the dump interface returns (lists per view)"""
    r = {}
    if pairs is not None:
        r["pairs_sha"] = sha(np.asarray(pairs, np.int64))
    for name, ms in (("scored", scored), ("kept", kept)):
        if ms is not None:
            r[f"{name}_n"] = np.array([len(m) for m in ms], np.int64)
            r[f"{name}_sha"] = sha(*[match_sha(m, exact_scores).encode() for m in ms])
            if not exact_scores:
                sc = np.concatenate([m["score3D"] for m in ms]).astype(np.float32)
                r[f"{name}_score_smp"] = sc[pick(len(sc))]
    if view_info is not None:
        r["view_info"] = np.array(view_info, np.float32)
    if estimates is not None:
        best, p = estimates
        r["est_n"] = np.int64(len(best))
        r["est_sha"] = match_sha(best, exact_scores)
        r["est_p_smp"] = np.asarray(p, np.float64)[pick(len(p))]
        if not exact_scores:
            r["est_score_smp"] = np.asarray(best["score3D"], np.float32)[pick(len(best))]
    if collinear is not None:
        r["collin_sha"] = sha(*[np.asarray(a, np.int64) for rp, idx in collinear for a in (rp, idx)])
    if l2g is not None:
        r["l2g_sha"] = sha(np.asarray(l2g, np.int64))
    for name, e in (("affraw", aff_raw), ("aff", aff)):
        if e is not None:
            r[f"{name}_n"] = np.int64(len(e[0]))
            r[f"{name}_idx_sha"] = sha(np.asarray(e[0], np.int64), np.asarray(e[1], np.int64))
            r[f"{name}_w_smp"] = np.asarray(e[2], np.float32)[pick(len(e[2]))]
    if num_lines is not None:
        r["num_lines"] = np.int64(num_lines)
    if residuals is not None:
        r["res_line_sha"] = sha(np.asarray(residuals["line"], np.int64))
        r["res_camseg_sha"] = sha(np.asarray(residuals["cam"], np.int64), np.asarray(residuals["seg"], np.int64))
    if segments is not None:
        r["seg_line_sha"] = sha(np.asarray(segments["line"], np.int64))
        pts = sorted_endpoints(segments)
        r["seg_n"] = np.int64(len(pts))
        r["seg_pts_smp"] = pts[pick(len(pts))]
    return r


def dump_record(P, cams, nsegs, matching=True, recon=True, collin=False, exact_scores=True):
    """stage_record of a pipeline with the dump interface of oracle/pyoracle.py (OraclePipeline, RefFullPipeline)"""
    kw = {}
    if matching:
        kw.update(pairs=P.pairs(), scored=[P.scored(c) for c in cams], kept=[P.matches(c) for c in cams],
                  view_info=[P.view_info(c) for c in cams], estimates=P.estimates())
    if collin:
        kw["collinear"] = [P.collinear(c, n) for c, n in zip(cams, nsegs)]
    if recon:
        kw.update(l2g=P.local2global(), aff_raw=P.affinity_raw(), aff=P.affinity(), num_lines=P.num_lines(), residuals=P.residuals(),
                  segments=P.segments3d())
    return stage_record(exact_scores=exact_scores, **kw)


def product_record(L, cams, nsegs, matching=True, recon=True, collin=False):
    """the same record of the product's L3DPP::Line3D mirror (line3dpp_b200.line3d.Line3D)"""
    kw = {}
    if matching:
        kw.update(pairs=L.pairs(), scored=[L.view_matches(c, kept_only=False) for c in cams], kept=[L.view_matches(c, kept_only=True) for c in cams],
                  view_info=[L.view_info(c) for c in cams], estimates=L.estimates())
    if collin:
        kw["collinear"] = [L.ctx_collinear(i, n) for i, n in enumerate(nsegs)]
    if recon:
        kw.update(l2g=L.local2global(), aff_raw=L.affinity(raw=True), aff=L.affinity(raw=False), num_lines=L.stats()["lines3D"],
                  residuals=L.residuals(), segments=L.segments3d())
    return stage_record(**kw)


def check_record(mine, ref, tol, skip=()):
    """exact equality of every key of the recorded reference except the sampled values (*_smp), which are compared with
    np.testing.assert_allclose(**tol[key]); keys in `skip` are not compared"""
    for k, v in ref.items():
        if k in skip:
            continue
        assert k in mine, k
        if k.endswith("_smp"):
            np.testing.assert_allclose(mine[k], v, err_msg=k, **tol[k])
        else:
            assert np.array_equal(np.asarray(mine[k]), np.asarray(v)), (k, mine[k], v)


def save_records(path, records):
    """records: {prefix: {key: value}} -> one .npz with keys prefix/key"""
    np.savez_compressed(path, **{f"{p}/{k}": np.asarray(v) for p, rec in records.items() for k, v in rec.items()})


def load_record(z, prefix):
    n = len(prefix) + 1
    return {k[n:]: (z[k][()] if z[k].ndim == 0 else z[k]) for k in z.files if k.startswith(prefix + "/")}


def rows_as_sets(counts, recs, fields=("tgt_seg", "overlap", "d_p1", "d_p2", "d_q1", "d_q2")):
    """per row: sorted list of tuples with float fields as raw bits"""
    out = []
    for r in range(len(counts)):
        row = []
        for i in range(counts[r]):
            e = recs[r, i]
            row.append(tuple(int(np.float32(e[f]).view(np.uint32)) if recs.dtype[f].kind == "f" else int(e[f]) for f in fields))
        out.append(sorted(row))
    return out


def two_view_scene(kind, n, seed):
    """two views of the same random 3D lines with an epipolar geometry the ring scenes do not have; kind = one of the named
    geometries or an explicit [(R, C), (R, C)] camera pair"""
    import dataclasses
    base = synth.make_scene(2, n, seed, "dense")
    rng = np.random.default_rng(seed)
    K = base.K[0]
    I = np.eye(3)
    rz = lambda a: np.array([[np.cos(a), -np.sin(a), 0], [np.sin(a), np.cos(a), 0], [0, 0, 1.0]])
    ry = lambda a: np.array([[np.cos(a), 0, np.sin(a)], [0, 1, 0], [-np.sin(a), 0, np.cos(a)]])
    cams = kind if not isinstance(kind, str) else {
            "sideways": [(I, (-0.3, 0.0, -4.0)), (I, (0.3, 0.0, -4.0))],            # epipole at infinity (E.z == 0), horizontal epipolar lines
            "forward": [(I, (0.0, 0.0, -4.6)), (I, (0.04, -0.03, -3.7))],            # epipole inside the image
            "edge": [(I, (0.0, 0.0, -4.2)), (ry(0.05), (0.9, 0.1, -3.6))],           # epipole a little outside the image border
            "rolled": [(I, (-0.4, 0.1, -4.0)), (rz(1.45) @ ry(-0.08), (0.5, -0.2, -4.1))]}[kind]
    P1, P2 = base.lines3d[:, :3], base.lines3d[:, 3:]
    Rs, ts, segs = [], [], []
    for R, C in cams:
        C = np.array(C)
        t = -R @ C
        X1, X2 = (R @ P1.T).T + t, (R @ P2.T).T + t
        u1 = X1[:, :2] / X1[:, 2:3] * synth.FOCAL + K[:2, 2] + rng.normal(scale=0.5, size=(len(P1), 2))
        u2 = X2[:, :2] / X2[:, 2:3] * synth.FOCAL + K[:2, 2] + rng.normal(scale=0.5, size=(len(P1), 2))
        ok = (X1[:, 2] > 0.1) & (X2[:, 2] > 0.1) & (np.linalg.norm(u1 - u2, axis=1) >= synth.MIN_LEN_PX)
        for u in (u1, u2):
            ok &= (u[:, 0] >= 0) & (u[:, 0] <= synth.WIDTH - 1) & (u[:, 1] >= 0) & (u[:, 1] <= synth.HEIGHT - 1)
        segs.append(np.ascontiguousarray(np.concatenate([u1, u2], axis=1)[ok][:n].astype(np.float32)))
        Rs.append(R); ts.append(t)
    return dataclasses.replace(base, R=np.array(Rs), t=np.array(ts), segs=segs)


def level1_scene(kind):
    """two_view_scene(kind, 1500, 31) plus horizontal / vertical / tiny segments and segments through the epipole"""
    sc = two_view_scene(kind, 1500, 31)
    rng = np.random.default_rng(5)
    for v in range(2):
        s = sc.segs[v]
        extra = []
        for _ in range(60):           # axis-parallel segments (parallel to the epipolar lines in the sideways case) and 1-2 px stubs
            x, y, l = rng.uniform(50, 2900), rng.uniform(50, 2200), rng.uniform(20, 400)
            extra += [(x, y, min(x + l, 3060), y), (x, y, x, min(y + l, 2290)), (x, y, x + 1.5, y + 0.5)]
        cx, cy = 1647.1, 1068.7                   # the epipole of the "forward" pair (0, 1): segments through / next to it
        for a in np.linspace(0, np.pi, 24, endpoint=False):
            extra += [(cx - 200 * np.cos(a), cy - 200 * np.sin(a), cx + 300 * np.cos(a), cy + 300 * np.sin(a)),
                      (cx + 3 * np.cos(a), cy + 3 * np.sin(a), cx + 150 * np.cos(a), cy + 150 * np.sin(a))]
        sc.segs[v] = np.ascontiguousarray(np.concatenate([s, np.array(extra, np.float32)]))
    return sc


def collinear_scene():
    """ring of 6 views with collinear fragments; view 3 ragged + degenerate, view 4 a single segment, view 5 empty"""
    from tests.golden.make_golden_collinear import edge_case_segments
    sc = synth.make_scene(6, 700, 92, "ring2", collinear=True)
    sc.segs[3] = np.ascontiguousarray(np.concatenate([edge_case_segments(), sc.segs[3][:37]]))
    sc.segs[4] = sc.segs[4][:1]
    sc.segs[5] = sc.segs[5][:0]
    return sc


def rdd_graph():
    """random symmetric affinity graph, every node with an edge"""
    rng = np.random.default_rng(3)
    n = 3000
    a = rng.integers(0, n, 40000); b = rng.integers(0, n, 40000)
    keep = a != b
    a, b = a[keep], b[keep]
    key = np.minimum(a, b) * n + np.maximum(a, b)
    _, idx = np.unique(key, return_index=True)
    a, b = a[np.sort(idx)], b[np.sort(idx)]
    missing = np.setdiff1d(np.arange(n), np.concatenate([a, b]))       # the reference kernel reads start index -1 otherwise
    a = np.concatenate([a, missing]); b = np.concatenate([b, (missing + 1) % n])
    w = rng.uniform(0.5, 1.0, len(a)).astype(np.float32)
    ei = np.stack([a, b], 1).reshape(-1).astype(np.int32)              # (i,j),(j,i) consecutive like A_
    ej = np.stack([b, a], 1).reshape(-1).astype(np.int32)
    return ei, ej, np.repeat(w, 2), n
