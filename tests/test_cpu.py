"""CPU-only tests (`pytest -m "not gpu"`): the oracle against the golden vectors produced by the UNMODIFIED reference
kernels on a B200 (tests/golden/), against the reference's clustering.cc compiled in place (runs on the CPU), the
oracle pipeline on synthetic scenes with known 3D lines, host-side sharding logic, and the C-ABI surface of the product
library (load + exported symbols; no compute without a GPU)."""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from line3dpp_b200 import synth
from tests import util

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden", "ref_kernels_v1.npz")
GOLD_REF_CPU = os.path.join(ROOT, "tests", "golden", "ref_outputs_cpu_v1.npz")


@pytest.fixture(scope="module")
def gold():
    if not os.path.exists(GOLD):
        pytest.skip("golden vectors not generated yet (tests/golden/make_golden.py on a GPU box)")
    return np.load(GOLD)


@pytest.fixture(scope="module")
def gscene(gold):
    v, n, seed = [int(x) for x in gold["scene_args"]]
    sc = synth.make_scene(v, n, seed, "dense")
    assert np.array_equal(np.stack(sc.segs), gold["segs"]), "synthetic scene generator changed: regenerate the golden file"
    return sc


# ---------------------------------------------------------------------------------------------- oracle vs golden
@pytest.mark.parametrize("tag,s,t", [("p01", 0, 1), ("p24", 2, 4)])
def test_oracle_match_dense_vs_reference_golden(oracle, gold, gscene, tag, s, t):
    g = lambda k: gold[f"{tag}_{k}"]
    dep, ov, _ = oracle.match_dense(oracle.lib().orc_match_dense_f32, gscene.segs[s], gscene.segs[t], g("F"), g("Rs"), g("Rt"), g("Cs"), g("Ct"), 0.25)
    assert np.array_equal(util.bits(ov), util.bits(g("dense_ov")))            # overlap: bit-exact on the CPU
    sel = g("dense_ov") > 0.25
    assert sel.sum() > 200
    rel = np.abs(dep[sel] - g("dense_dep")[sel]) / np.maximum(np.abs(g("dense_dep")[sel]), 1e-3)
    assert np.median(rel) < 1e-6 and np.quantile(rel, 0.999) < 1e-2          # depths: host rsqrt vs MUFU.RSQ
    assert np.array_equal(dep[~sel], g("dense_dep")[~sel])                   # -1 everywhere else


@pytest.mark.parametrize("tag,s,t", [("p01", 0, 1), ("p24", 2, 4)])
def test_oracle_knn_lists_vs_reference_golden(oracle, gold, gscene, tag, s, t):
    g = lambda k: gold[f"{tag}_{k}"]
    counts, out, total, _ = oracle.match_lines(oracle.lib().orc_match_lines_f32, gscene.segs[s], gscene.segs[t], g("F"), g("Rs"), g("Rt"), g("Cs"), g("Ct"), s, t, 0.25, 10)
    assert np.array_equal(counts, g("knn_counts")) and total == g("knn_counts").sum()
    ref = g("knn")
    for r in range(len(counts)):
        a, b = out[r, :counts[r]], ref[r, :counts[r]]
        assert np.array_equal(a["tgt_seg"], b["tgt_seg"]) and np.array_equal(util.bits(a["overlap"]), util.bits(b["overlap"]))


def test_oracle_scores_vs_reference_golden(oracle, gold, gscene):
    p = gold["score_params"]
    scores, _ = oracle.score_matches(oracle.lib().orc_score_matches_f32, gscene.segs[0], gold["score_m4"], gold["score_ranges"], gold["score_reg"],
                                     gold["score_R"], gold["score_C"], float(p[0]), float(p[1]), float(p[2]))
    ref = gold["score_out"]
    assert len(ref) > 1000 and (ref > 0).sum() > 100
    off = ~np.isclose(scores, ref, rtol=1e-4, atol=1e-5)
    assert off.mean() < 5e-3       # a similarity at the 0.5 truncation may flip with a 1-ulp expf/acosf difference
    assert np.median(np.abs(scores - ref)) < 1e-6


def test_oracle_rdd_vs_reference_golden(oracle, gold):
    n = int(gold["rdd_n"][0])
    oi, oj, ow, _ = oracle.rdd(oracle.lib().orc_rdd_f32, gold["rdd_ei"], gold["rdd_ej"], gold["rdd_ew"], n)
    assert np.array_equal(oi, gold["rdd_oi"]) and np.array_equal(oj, gold["rdd_oj"])
    assert np.array_equal(util.bits(ow), util.bits(gold["rdd_ow"]))           # + - * / only: bit-exact


def test_oracle_cluster_vs_reference_golden(oracle, gold):
    n = int(gold["rdd_n"][0])
    lab = oracle.cluster(oracle.lib().orc_cluster, gold["rdd_ei"], gold["rdd_ej"], gold["rdd_ew"], n)
    assert np.array_equal(lab, gold["cluster_labels"])
    lab2 = oracle.cluster(oracle.lib().orc_cluster, gold["rdd_oi"], gold["rdd_oj"], gold["rdd_ow"], n)
    assert np.array_equal(lab2, gold["cluster_labels_rdd"])


def test_oracle_cluster_vs_reference_clustering_cc_live(oracle):
    """the reference's clustering.cc on random graphs (labels recorded by tests/golden/make_ref_outputs.py)"""
    z = np.load(GOLD_REF_CPU)
    rng = np.random.default_rng(1)
    for n, m in [(10, 30), (500, 4000), (2000, 3000)]:
        ei, ej = rng.integers(0, n, m).astype(np.int32), rng.integers(0, n, m).astype(np.int32)
        ew = rng.choice(np.linspace(0.5, 1.0, 23), m).astype(np.float32)     # many ties: stable-sort order matters
        a = oracle.cluster(oracle.lib().orc_cluster, ei, ej, ew, n)
        assert np.array_equal(a, util.load_record(z, f"cluster_live/{n}_{m}")["labels"])


# ---------------------------------------------------------------------------------------------- oracle pipeline sanity
def _dist_to_gt(pts, gt):
    a = gt[:, :3]
    d = gt[:, 3:] - a
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    w = pts[:, None, :] - a[None]
    return np.linalg.norm(w - (w * d[None]).sum(-1, keepdims=True) * d[None], axis=-1).min(1)


@pytest.mark.parametrize("use_gpu,diffusion", [(1, False), (1, True), (0, False)])
def test_oracle_pipeline_recovers_ground_truth_lines(oracle, use_gpu, diffusion):
    sc = synth.make_scene(10, 250, 9, "ring3")
    P = oracle.OraclePipeline(False, use_gpu)
    P.add_scene(sc)
    assert P.match_images() == 0
    assert P.pair_evals() == sum(len(sc.segs[s]) * len(sc.segs[t]) for s, t in synth.view_pairs(sc.neighbors))
    assert np.array_equal(P.pairs(), synth.view_pairs(sc.neighbors))
    assert P.reconstruct(3, diffusion) == 0
    s = P.segments3d()
    assert P.num_lines() > 150
    assert np.median(_dist_to_gt(s["p1"], sc.lines3d)) < 5e-3 and np.median(_dist_to_gt(s["p2"], sc.lines3d)) < 5e-3


def test_oracle_gpu_and_cpu_semantics_agree_statistically(oracle):
    sc = synth.make_scene(10, 250, 9, "ring3")
    n = []
    for use_gpu in (1, 0):
        P = oracle.OraclePipeline(False, use_gpu)
        P.add_scene(sc)
        P.match_images()
        P.reconstruct(3, False)
        n.append(P.num_lines())
    assert abs(n[0] - n[1]) <= 0.05 * n[0]


def test_oracle_edge_cases(oracle):
    L = oracle.lib()
    P = oracle.OraclePipeline(False, 1)
    K = np.array([[1000., 0, 500], [0, 1000., 400], [0, 0, 1]])
    seg = np.array([[10, 10, 100, 100]], np.float32)
    assert P.add_view(0, 600, 400, K, np.eye(3), np.zeros(3), 1.0, [1], seg) == -1     # image too small (line3D.cc:119)
    assert P.add_view(0, 1000, 800, K, np.eye(3), np.zeros(3), 1.0, [], seg) == -3      # no neighbours (line3D.cc:154)
    assert P.add_view(0, 1000, 800, K, np.eye(3), np.zeros(3), 1.0, [1], seg) == 0
    assert P.add_view(0, 1000, 800, K, np.eye(3), np.zeros(3), 1.0, [1], seg) == -2     # duplicate id (line3D.cc:130)
    assert P.match_images() == 0                                                        # neighbour 1 does not exist: nothing to match
    assert P.reconstruct(3, False) == -1                                                # no estimates (line3D.cc:1712)
    # degenerate geometry: identical cameras -> F = 0 -> every intersection invalid -> no matches, no crash
    z = np.zeros(9, np.float32)
    c, o, tot, _ = oracle.match_lines(L.orc_match_lines_f32, seg, seg, z, np.eye(3, dtype=np.float32).ravel(), np.eye(3, dtype=np.float32).ravel(),
                                      np.zeros(3, np.float32), np.zeros(3, np.float32), 0, 1, 0.25, 10)
    assert tot == 0


# ---------------------------------------------------------------------------------------------- host logic
def test_view_pairs_follow_reference_order():
    nb = [np.array([1, 2], np.uint32), np.array([0], np.uint32), np.array([3], np.uint32), np.array([0, 2], np.uint32)]
    assert synth.view_pairs(nb).tolist() == [[0, 1], [0, 2], [2, 3], [3, 0]]
    assert len(synth.view_pairs(synth.ring_neighbors(1000, 5))) == 5000
    assert len(synth.view_pairs(synth.dense_neighbors(200))) == 19900


def test_scene_shards_are_consistent():
    full = synth.make_scene(12, 100, 4, "ring2")
    part = synth.make_scene_views(12, 100, 4, "ring2", [3, 4, 5])
    for v in (3, 4, 5):
        assert np.array_equal(full.segs[v], part.segs[v])
    assert len(part.segs[0]) == 0 and np.array_equal(full.K, part.K) and np.array_equal(full.R, part.R)



# ---------------------------------------------------------------------------------------------- collinearity (SURVEY §8f-3)
GOLD_COLLIN = os.path.join(ROOT, "tests", "golden", "ref_collinear_v1.npz")


@pytest.mark.parametrize("name", ["v0", "v2", "edge"])
def test_oracle_collinear_vs_reference_golden(oracle, name):
    """orc_collinear_f32 == the UNMODIFIED K_collinearity run on a B200 (tests/golden/make_golden_collinear.py)"""
    if not os.path.exists(GOLD_COLLIN):
        pytest.skip("collinearity golden vectors not generated yet (tests/golden/make_golden_collinear.py on a GPU box)")
    g = np.load(GOLD_COLLIN)
    segs = g[f"{name}_segs"]
    if name != "edge":
        v, n, seed = [int(x) for x in g["scene_args"]]
        sc = synth.make_scene(v, n, seed, "ring1", collinear=True)
        assert np.array_equal(sc.segs[int(name[1:])], segs), "synthetic scene generator changed: regenerate the golden file"
    for t in (0.5, 2.0, 6.0):
        Cm, _ = oracle.collinear(oracle.lib().orc_collinear_f32, segs, t)
        assert np.array_equal(np.argwhere(Cm == 1).astype(np.int32), g[f"{name}_t{t}"]), (name, t)


def test_oracle_collinear_properties(oracle):
    """symmetric, empty diagonal, monotone in the threshold, float and double paths agree on well-conditioned input,
    and the fragments of a broken 3D line are found"""
    sc = synth.make_scene(4, 300, 95, "ring1", collinear=True)
    L = oracle.lib()
    prev = None
    for t in (1.0, 2.0, 5.0):
        a, _ = oracle.collinear(L.orc_collinear_f32, sc.segs[1], t)
        b, _ = oracle.collinear(L.orc_collinear_f64, sc.segs[1], t)
        assert np.array_equal(a, a.T) and not a.diagonal().any() and np.array_equal(a, b)
        if prev is not None:
            assert np.all(a >= prev)
        prev = a
    ids = sc.line_ids[1]
    frag = {(i, j) for i in range(len(ids)) for j in range(len(ids)) if i != j and ids[i] // 2 == ids[j] // 2}
    found = {tuple(x) for x in np.argwhere(prev == 1)}
    assert len(frag) > 20 and len(frag & found) >= 0.9 * len(frag)
    e, _ = oracle.collinear(L.orc_collinear_f32, np.zeros((0, 4), np.float32), 2.0)
    assert e.shape == (0, 0)


@pytest.mark.parametrize("use_gpu", [1, 0])
def test_oracle_collinearity_links_merge_fragments(oracle, use_gpu):
    sc = synth.make_scene(8, 300, 3, "ring2", collinear=True)
    out = {}
    for ct in (-1.0, 2.0):
        P = oracle.OraclePipeline(False, use_gpu)
        P.add_scene(sc)
        P.match_images()
        assert P.reconstruct(3, bool(use_gpu), ct) == 0
        out[ct] = (P.num_lines(), len(P.affinity_raw()[0]), sum(len(P.collinear(c, len(s))[1]) for c, s in zip(sc.cam_ids, sc.segs)))
        s = P.segments3d()
        assert np.median(_dist_to_gt(s["p1"], sc.lines3d)) < 5e-3
    assert out[-1.0][2] == 0 and out[2.0][2] > 300
    assert out[2.0][1] > out[-1.0][1] and out[2.0][0] < out[-1.0][0]


# ---------------------------------------------------------------------------------------------- line bundling (SURVEY §8f-4)
def _np_cost(x, cams, rc, xy):
    """independent numpy restatement of the bundling cost of ONE line (optimization.h:66-162 + HuberLoss(2)), no derivatives"""
    om, s = x[0], x[1:]
    nm = s @ s
    sx = np.array([[0, -s[2], s[1]], [s[2], 0, -s[0]], [-s[1], s[0], 0]])
    Q = ((1 - nm) * np.eye(3) + 2 * sx + 2 * np.outer(s, s)) / (1 + nm)
    l, m = Q[:, 0], om * Q[:, 1]
    c = 0.0
    for cam, o in zip(rc, xy):
        R, C, fx, fy, px, py = cams[cam, :9].reshape(3, 3), cams[cam, 9:12], *cams[cam, 12:16]
        q = R @ (m - np.cross(C, l))
        pl = np.array([fy * q[0], fx * q[1], -fy * px * q[0] - fx * py * q[1] + fx * fy * q[2]])
        d = np.hypot(pl[0], pl[1])
        dr = (o[2:] - o[:2]) / np.linalg.norm(o[2:] - o[:2])
        ang = np.arccos(np.clip((pl[0] * -dr[1] + pl[1] * dr[0]) / d, -1, 1))
        ang = min(ang, np.pi - ang)
        r = np.array([pl[0] * o[0] + pl[1] * o[1] + pl[2], pl[0] * o[2] + pl[1] * o[3] + pl[2]]) / d * np.exp(2 * ang)
        sq = r @ r
        c += 0.5 * (sq if sq <= 4 else 4 * np.sqrt(sq) - 4)
    return c


def test_oracle_optimizer_vs_reference_ceres_fixture(oracle):
    """orc_optimize_lines from the reference's UNOPTIMISED result lines + residuals reproduces the reference's own
    OPTIMIZED result (testdata/Line3D++_ref, both files; 2489 clusters with identical residual sets).  The fixture text has
    ~5e-6 of rounding; LineOptimizer moves the lines by 3.8e-4 (median), up to 1.6e-2."""
    from tests import nvm_util as nu
    before, after, ptr, res = nu.load_opt_pairs()
    cams, shift = nu.optimizer_inputs(nu.load_inputs())
    b = before + np.tile(shift, 2)
    out, valid, summ = oracle.optimize_lines(oracle.lib().orc_optimize_lines, b, ptr, res[:, 0].astype(np.int32), res[:, 2:6], cams, 250)
    out -= np.tile(shift, 2)
    assert valid.all() and summ[3] == 0 and summ[5] == len(before)              # converged, every line free
    assert summ[2] < 0.85 * summ[1]                                             # total cost 9514 -> ~7950
    moved, gap = nu.line_gap(after, before), nu.line_gap(after, out)
    assert np.median(moved) > 3e-4
    assert np.median(gap) < 2.5e-5 and np.percentile(gap, 90) < 1.5e-4 and np.percentile(gap, 99) < 8e-4, (np.median(gap), np.percentile(gap, [90, 99]))
    big = moved > 1e-3                                                           # where the reference really moved a line we follow it
    assert big.sum() > 200 and np.median(gap[big] / moved[big]) < 0.05


def test_oracle_optimizer_reaches_a_minimum_of_the_independent_cost(oracle):
    """the final Cayley parameters minimise an INDEPENDENT numpy restatement of the robust cost: scipy cannot improve them"""
    from scipy.optimize import minimize
    from tests import nvm_util as nu
    before, after, ptr, res = nu.load_opt_pairs()
    cams, shift = nu.optimizer_inputs(nu.load_inputs())
    sel = np.arange(0, 600, 20)
    b = (before + np.tile(shift, 2))[sel]
    p2 = np.concatenate([[0], np.cumsum(np.diff(ptr)[sel])])
    rr = np.concatenate([res[ptr[i]:ptr[i + 1]] for i in sel])
    out, valid, summ = oracle.optimize_lines(oracle.lib().orc_optimize_lines, b, p2, rr[:, 0].astype(np.int32), rr[:, 2:6], cams, 250)

    def cayley(seg):                                   # optimization.cc:34-70
        l = (seg[3:] - seg[:3]) / np.linalg.norm(seg[3:] - seg[:3])
        m = np.cross(0.5 * (seg[:3] + seg[3:]), l)
        Q = np.stack([l, m / np.linalg.norm(m), np.cross(l, m) / np.linalg.norm(np.cross(l, m))], 1)
        S = (Q - np.eye(3)) @ np.linalg.inv(Q + np.eye(3))
        return np.array([np.linalg.norm(m), S[2, 1], S[0, 2], S[1, 0]])
    tot0 = tot1 = tot2 = 0.0
    for k in range(len(sel)):
        rc, xy = rr[p2[k]:p2[k + 1], 0].astype(int), rr[p2[k]:p2[k + 1], 2:6]
        x0, x1 = cayley(b[k]), cayley(out[k])
        c0, c1 = _np_cost(x0, cams, rc, xy), _np_cost(x1, cams, rc, xy)
        c2 = minimize(_np_cost, x1, args=(cams, rc, xy), method="Nelder-Mead", options=dict(xatol=1e-10, fatol=1e-12, maxiter=2000)).fun
        tot0 += c0; tot1 += c1; tot2 += c2
    assert abs(tot0 - summ[1]) < 1e-6 * tot0 and abs(tot1 - summ[2]) < 1e-6 * tot1        # same cost function, independently coded
    # Ceres stops on the relative change of the TOTAL cost (function_tolerance 1e-6), so single lines keep a little slack
    assert tot1 < 0.85 * tot0 and tot1 - tot2 < 1e-3 * tot1


def test_oracle_optimizer_edge_cases(oracle):
    fn = oracle.lib().orc_optimize_lines
    cams = np.zeros((1, 16)); cams[0, [0, 4, 8]] = 1; cams[0, 12:16] = (1000, 1000, 500, 400)
    seg = np.array([[0.3, 0.2, 5.0, 0.8, 0.25, 5.5]])
    # a line without residuals, and max_iter = 0, stay where they are (unit direction around the old mid point)
    for ptr, it in (([0, 0], 250), ([0, 1], 0)):
        out, valid, summ = oracle.optimize_lines(fn, seg, ptr, [0] * ptr[1], np.array([[100., 100, 300, 120]] * ptr[1]).reshape(-1, 4), cams, it)
        mid = 0.5 * (seg[0, :3] + seg[0, 3:])
        assert valid[0] == 1 and np.allclose(0.5 * (out[0, :3] + out[0, 3:]), mid, atol=1e-9) and abs(np.linalg.norm(out[0, :3] - out[0, 3:]) - 2) < 1e-9
        d = (seg[0, 3:] - seg[0, :3]) / np.linalg.norm(seg[0, 3:] - seg[0, :3])
        assert abs(abs(((out[0, :3] - out[0, 3:]) / 2) @ d) - 1) < 1e-9
    out, valid, summ = oracle.optimize_lines(fn, np.zeros((0, 6)), [0], [], np.zeros((0, 4)), cams, 10)
    assert len(out) == 0


@pytest.mark.parametrize("use_gpu", [1, 0])
def test_oracle_pipeline_with_bundling(oracle, use_gpu):
    sc = synth.make_scene(10, 250, 9, "ring3", noise_px=1.0)
    d = {}
    for uc in (False, True):
        P = oracle.OraclePipeline(False, use_gpu)
        P.add_scene(sc); P.match_images()
        assert P.reconstruct(3, False, -1.0, uc) == 0
        s = P.segments3d()
        d[uc] = (P.num_lines(), np.mean(np.concatenate([_dist_to_gt(s["p1"], sc.lines3d), _dist_to_gt(s["p2"], sc.lines3d)])))
        if uc:
            sm = P.opt_summary()
            assert sm[3] == 0 and sm[2] < sm[1] and sm[5] > 100
    assert abs(d[True][0] - d[False][0]) <= 2 and d[True][1] < d[False][1]          # closer to the ground-truth lines


# ---------------------------------------------------------------------------------------------- cluster -> 3D segments (SURVEY §8f-1)
def test_oracle_cluster_tail_reproduces_the_reference_result_file(oracle):
    """findCollinearSegments(cluster) + project2DsegmentOnto3Dline (line3D.cc:2221-2266, 2342-2452) on the reference's OWN
    clusters: from the line and the 2D residuals listed in testdata/Line3D++_ref/*.txt the oracle rebuilds every one of the
    2501 3D segments of that file (end points to the text rounding); the few extra segments are the tiny ones the
    reference removes afterwards (filterTinySegments needs the cluster's reference view, which the file does not record)."""
    from tests import nvm_util as nu
    inp = nu.load_inputs()
    cam_segs, clusters = nu.fixture_clusters()
    P = oracle.OraclePipeline(True, 1)
    for i in range(inp["V"]):
        w, h = inp["wh"][i]
        assert P.add_view(i, int(w), int(h), inp["K"][i], inp["R"][i], inp["t"][i], inp["median_depth"][i], inp["wps"][i], cam_segs[i]) == 0
    out = np.zeros((64, 6))
    L = oracle.lib()

    def run(cl):
        n = L.orc_collinear_from_cluster(P.ctx, oracle._p(np.ascontiguousarray(cl["p1p2"])), len(cl["cams"]), oracle._p(cl["cams"]), oracle._p(cl["segs"]),
                                         oracle._p(out), 64)
        return out[:n].copy()
    total, matched, extra, worst = nu.check_fixture_segments(run, clusters)
    assert total == 2501 and matched == total and worst < 5e-5, (total, matched, worst)
    assert extra <= 0.02 * total, extra


# ---------------------------------------------------------------------------------------------- .nvm input format (SURVEY §8f-2)
def _read_nvm_product(path):
    from line3dpp_b200 import build
    L = ctypes.CDLL(build.build())
    L.l3dpp_nvm_open.restype = ctypes.c_void_p
    err = ctypes.create_string_buffer(256)
    h = L.l3dpp_nvm_open(str(path).encode(), err, 256)
    if not h:
        return None, err.value.decode()
    h = ctypes.c_void_p(h)
    cams = []
    for i in range(L.l3dpp_nvm_num_cameras(h)):
        R, t, Cc = np.zeros(9), np.zeros(3), np.zeros(3)
        f, d, md, nw = ctypes.c_float(), ctypes.c_float(), ctypes.c_float(), ctypes.c_int()
        name = ctypes.create_string_buffer(512)
        p = lambda a: a.ctypes.data_as(ctypes.c_void_p)
        assert L.l3dpp_nvm_camera(h, i, p(R), p(t), p(Cc), ctypes.byref(f), ctypes.byref(d), ctypes.byref(md), ctypes.byref(nw), name, 512) == 0
        w = np.zeros(max(nw.value, 1), np.uint32)
        assert L.l3dpp_nvm_worldpoints(h, i, p(w), nw.value) == nw.value
        cams.append(dict(R=R.reshape(3, 3), t=t, C=Cc, f=f.value, dist=d.value, md=md.value, wps=w[:nw.value], name=name.value.decode()))
    L.l3dpp_nvm_close(h)
    return cams, ""


def test_nvm_reader_round_trip(tmp_path):
    """L3DPP::readNVM (include/line3d_io.h; restates main_vsfm.cpp:143-310) on a synthetic NVM_V3 model"""
    rng = np.random.default_rng(3)
    V, NP = 5, 40
    q = rng.normal(size=(V, 4)); q /= np.linalg.norm(q, axis=1, keepdims=True)
    Cc = rng.uniform(-3, 3, (V, 3)); f = rng.uniform(800, 2500, V); d = np.array([0, 0.01, 0, -0.02, 0])
    pts = rng.uniform(-1, 1, (NP, 3))
    vis = [sorted(rng.choice(V, size=rng.integers(2, V + 1), replace=False).tolist()) for _ in range(NP)]
    lines = ["NVM_V3", "", str(V)]
    for i in range(V):
        lines.append(f"dir/img{i}.jpg\t{f[i]:.10f} {q[i,0]:.12f} {q[i,1]:.12f} {q[i,2]:.12f} {q[i,3]:.12f} {Cc[i,0]:.12f} {Cc[i,1]:.12f} {Cc[i,2]:.12f} {d[i]:.6f} 0")
    lines += ["", str(NP)]
    for j in range(NP):
        meas = " ".join(f"{c} {7 * j + c} {10.5 + c} {-3.25 + j}" for c in vis[j])
        lines.append(f"{pts[j,0]:.12f} {pts[j,1]:.12f} {pts[j,2]:.12f} 255 128 0 {len(vis[j])} {meas}")
    path = tmp_path / "model.nvm"
    path.write_text("\n".join(lines) + "\n0\n")
    cams, err = _read_nvm_product(path)
    assert cams is not None, err
    assert len(cams) == V
    for i, c in enumerate(cams):
        qw, qx, qy, qz = [float(f"{v:.12f}") for v in q[i]]
        R = np.array([[1 - 2 * qy * qy - 2 * qz * qz, 2 * qx * qy - 2 * qz * qw, 2 * qx * qz + 2 * qy * qw],
                      [2 * qx * qy + 2 * qz * qw, 1 - 2 * qx * qx - 2 * qz * qz, 2 * qy * qz - 2 * qx * qw],
                      [2 * qx * qz - 2 * qy * qw, 2 * qy * qz + 2 * qx * qw, 1 - 2 * qx * qx - 2 * qy * qy]])
        Ci = np.array([float(f"{v:.12f}") for v in Cc[i]])
        np.testing.assert_allclose(c["R"], R, atol=1e-14)
        np.testing.assert_allclose(c["t"], -R @ Ci, atol=1e-13)
        assert c["name"] == f"dir/img{i}.jpg" and abs(c["f"] - np.float32(f[i])) < 1e-3 and abs(c["dist"] - d[i]) < 1e-7
        mine = [j for j in range(NP) if i in vis[j]]
        assert c["wps"].tolist() == mine
        dep = np.sort(np.array([np.float32(np.linalg.norm(np.array([float(f"{v:.12f}") for v in pts[j]]) - Ci)) for j in mine], np.float32))
        assert c["md"] == (dep[len(dep) // 2] if len(dep) else 0.0)
    bad, err = _read_nvm_product(tmp_path / "missing.nvm")
    assert bad is None and "cannot open" in err
    (tmp_path / "empty.nvm").write_text("NVM_V3\n\n0\n")
    bad, err = _read_nvm_product(tmp_path / "empty.nvm")
    assert bad is None and "No aligned cameras" in err


def test_nvm_reader_on_the_reference_test_data(tmp_path):
    """readNVM on the reference's own testdata/vsfm_result.nvm (every camera, a seeded sample of 500 of its 3D points; see
    tests/golden/make_nvm_inputs.py --sample): cameras equal the committed inputs of the nvm configuration, world points and
    median depths equal the restatement that produced those inputs"""
    import gzip
    from tests import nvm_util as nu
    from tests.golden.make_nvm_inputs import read_nvm
    path = tmp_path / "vsfm_result.nvm"
    path.write_bytes(gzip.open(os.path.join(ROOT, "tests", "golden", "vsfm_result_sample_v1.nvm.gz")).read())
    inp = nu.load_inputs()
    cams, err = _read_nvm_product(path)
    assert cams is not None and len(cams) == inp["V"], err
    _, wps, depths = read_nvm(str(path))
    from line3dpp_b200 import build
    L = ctypes.CDLL(build.build())
    for i, c in enumerate(cams):
        np.testing.assert_allclose(c["R"], inp["R"][i], atol=1e-15)
        np.testing.assert_allclose(c["t"], inp["t"][i], atol=1e-13)
        d = np.sort(np.array(depths[i], np.float32))
        assert c["md"] == (d[len(d) // 2] if len(d) else 0.0) and c["wps"].tolist() == wps[i]
        K = np.zeros(9)
        L.l3dpp_intrinsics_from_focal(ctypes.c_float(c["f"]), int(inp["wh"][i][0]), int(inp["wh"][i][1]), K.ctypes.data_as(ctypes.c_void_p))
        assert np.array_equal(K.reshape(3, 3), inp["K"][i])
    assert sum(len(w) for w in wps) > 1000

# ---------------------------------------------------------------------------------------------- product library surface
def test_capi_library_loads_and_exports_every_declared_symbol():
    from line3dpp_b200 import build
    so = build.build()
    lib = ctypes.CDLL(so)
    hdr = open(os.path.join(ROOT, "include", "l3d_capi.h")).read()
    names = sorted(set(re.findall(r"\b(l3d_[a-z0-9_]+)\s*\(", hdr)))
    assert len(names) >= 20
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/l3d_capi.h but not exported"
    for n in ("l3dpp_create", "l3dpp_add_image", "l3dpp_match_images", "l3dpp_reconstruct", "l3dpp_save_txt"):
        assert hasattr(lib, n)


def test_nvm_reader_rejects_truncated_camera_list(tmp_path):
    """ADVICE r1: a truncated camera section must be an error, not a default camera"""
    f = tmp_path / "t.nvm"
    f.write_text("NVM_V3\n\n3\nimg0.jpg 1000 1 0 0 0 0 0 0 0 0\nimg1.jpg 1000 1 0 0 0\n")
    cams, err = _read_nvm_product(f)
    assert cams is None and "camera" in err
    f.write_text("NVM_V3\n\n2\nimg0.jpg 1000 1 0 0 0 0 0 0 0 0\n")
    cams, err = _read_nvm_product(f)
    assert cams is None and "end of file" in err


def _read_sfm_product(kind, path, aux=""):
    from line3dpp_b200 import build
    L = ctypes.CDLL(build.build())
    L.l3dpp_sfm_open.restype = ctypes.c_void_p
    err = ctypes.create_string_buffer(256)
    h = L.l3dpp_sfm_open(kind, str(path).encode(), str(aux).encode(), err, 256)
    if not h:
        return None, err.value.decode()
    h = ctypes.c_void_p(h)
    p = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    cams = []
    for i in range(L.l3dpp_sfm_num_cameras(h)):
        head, K, R, t, Cc, dist = np.zeros(5), np.zeros(9), np.zeros(9), np.zeros(3), np.zeros(3), np.zeros(5)
        name = ctypes.create_string_buffer(512)
        assert L.l3dpp_sfm_camera(h, i, p(head), p(K), p(R), p(t), p(Cc), p(dist), name, 512) == 0
        w = np.zeros(max(int(head[4]), 1), np.uint32)
        assert L.l3dpp_sfm_worldpoints(h, i, p(w), int(head[4])) == int(head[4])
        cams.append(dict(id=int(head[0]), has_K=bool(head[1]), f=head[2], md=np.float32(head[3]), wps=w[:int(head[4])], K=K.reshape(3, 3), R=R.reshape(3, 3),
                         t=t, C=Cc, dist=dist, name=name.value.decode()))
    L.l3dpp_sfm_close(h)
    return cams, ""


def _rot(rng):
    q = rng.normal(size=4); q /= np.linalg.norm(q)
    w, x, y, z = q
    return q, np.array([[1 - 2 * y * y - 2 * z * z, 2 * x * y - 2 * z * w, 2 * x * z + 2 * y * w], [2 * x * y + 2 * z * w, 1 - 2 * x * x - 2 * z * z, 2 * y * z - 2 * x * w],
                        [2 * x * z - 2 * y * w, 2 * y * z + 2 * x * w, 1 - 2 * x * x - 2 * y * y]])


def test_bundler_reader(tmp_path):
    """L3DPP::readBundler (include/line3d_io.h; restates main_bundler.cpp:143-286) on a synthetic bundle.rd.out"""
    rng = np.random.default_rng(5)
    V, NP = 4, 30
    Rs = [_rot(rng)[1] for _ in range(V)]; ts = rng.uniform(-2, 2, (V, 3)); f = rng.uniform(500, 2000, V); k = rng.uniform(-0.1, 0.1, (V, 2))
    pts = rng.uniform(-1, 1, (NP, 3))
    vis = [sorted(rng.choice(V, size=rng.integers(2, V + 1), replace=False).tolist()) for _ in range(NP)]
    L = ["# Bundle file v0.3", f"{V} {NP}"]
    for i in range(V):
        L.append(f"{f[i]:.10f} {k[i,0]:.10f} {k[i,1]:.10f}")
        L += [" ".join(f"{v:.12f}" for v in Rs[i][r]) for r in range(3)]
        L.append(" ".join(f"{v:.12f}" for v in ts[i]))
    for j in range(NP):
        L += [" ".join(f"{v:.12f}" for v in pts[j]), "255 0 0", f"{len(vis[j])} " + " ".join(f"{c} {j} 1.5 -2.5" for c in vis[j])]
    (tmp_path / "bundle.rd.out").write_text("\n".join(L) + "\n")
    (tmp_path / "list.txt").write_text("a.jpg 0 123\nb.jpg\n\nd.jpg 1 2\n")
    cams, err = _read_sfm_product(0, tmp_path / "bundle.rd.out", tmp_path / "list.txt")
    assert cams is not None and len(cams) == V, err
    rd = lambda a: np.array([float(f"{v:.12f}") for v in np.ravel(a)]).reshape(np.shape(a))
    for i, c in enumerate(cams):
        R = rd(Rs[i]); R[1:] *= -1
        t = rd(ts[i]); t[1:] *= -1
        np.testing.assert_allclose(c["R"], R, atol=1e-15); np.testing.assert_allclose(c["t"], t, atol=1e-15)
        Ci = -R.T @ t
        np.testing.assert_allclose(c["C"], Ci, atol=1e-14)
        assert c["id"] == i and not c["has_K"] and abs(c["f"] - np.float32(float(f"{f[i]:.10f}"))) < 1e-3
        np.testing.assert_allclose(c["dist"][:2], np.float32(rd(k[i])), atol=1e-9); assert not c["dist"][2:].any()
        mine = [j for j in range(NP) if i in vis[j]]
        assert c["wps"].tolist() == mine
        dep = np.sort(np.array([np.float32(np.linalg.norm(rd(pts[j]) - c["C"])) for j in mine], np.float32))
        assert c["md"] == (dep[len(dep) // 2] if len(dep) else np.float32(0))
    assert [c["name"] for c in cams] == ["a.jpg", "b.jpg", "", "d.jpg"]
    (tmp_path / "empty.out").write_text("# Bundle file v0.3\n0 0\n")
    bad, err = _read_sfm_product(0, tmp_path / "empty.out")
    assert bad is None and "No cameras" in err


def test_colmap_reader(tmp_path):
    """L3DPP::readColmap (include/line3d_io.h; restates main_colmap.cpp:140-401) on a synthetic text model"""
    rng = np.random.default_rng(6)
    cam_lines = ["# Camera list", "1 SIMPLE_PINHOLE 640 480 500.5 320 240", "2 PINHOLE 640 480 500 510 321 239", "3 SIMPLE_RADIAL 640 480 400 300 200 0.01",
                 "4 RADIAL 640 480 410 310 210 0.02 -0.03", "5 OPENCV 800 600 700 710 400 300 0.1 0.2 0.001 0.002",
                 "6 FULL_OPENCV 800 600 701 711 401 301 0.11 0.21 0.0011 0.0021 0.31 0 0 0"]
    (tmp_path / "cameras.txt").write_text("\n".join(cam_lines) + "\n")
    NP = 25
    pts = rng.uniform(-1, 1, (NP, 3))
    imgs, L = [], ["# Image list with two lines of data per image:"]
    for n, (img_id, cam_id) in enumerate([(10, 1), (11, 2), (12, 3), (13, 4), (14, 5), (15, 6), (16, 99)]):
        q, R = _rot(rng)
        q = q * 1.7                                   # rotationFromQ normalises (line3D.cc:2737-2754)
        t = rng.uniform(-2, 2, 3)
        seen = sorted(rng.choice(NP, size=8, replace=False).tolist())
        obs = " ".join(f"{1.0 + j} {2.0 + j} {(-1 if k % 3 == 0 else p)}" for k, (j, p) in enumerate(zip(range(8), seen)))
        L += [f"{img_id} {q[0]:.12f} {q[1]:.12f} {q[2]:.12f} {q[3]:.12f} {t[0]:.12f} {t[1]:.12f} {t[2]:.12f} {cam_id} im{img_id}.png", obs]
        imgs.append((img_id, cam_id, q, t, [p for k, p in enumerate(seen) if k % 3 != 0]))
    (tmp_path / "images.txt").write_text("\n".join(L) + "\n")
    (tmp_path / "points3D.txt").write_text("# 3D point list\n" + "\n".join(f"{j} {pts[j,0]:.12f} {pts[j,1]:.12f} {pts[j,2]:.12f} 1 2 3 0.5 10 1" for j in range(NP) if j != 7) + "\n")
    cams, err = _read_sfm_product(1, tmp_path)
    assert cams is not None, err
    assert [c["id"] for c in cams] == [10, 11, 12, 13, 14, 15]                     # image 16 uses an unknown camera: dropped
    expK = {1: (500.5, 500.5, 320, 240), 2: (500, 510, 321, 239), 3: (400, 400, 300, 200), 4: (410, 410, 310, 210), 5: (700, 710, 400, 300), 6: (701, 711, 401, 301)}
    expD = {1: (0, 0, 0, 0, 0), 2: (0, 0, 0, 0, 0), 3: (0.01, 0, 0, 0, 0), 4: (0.02, -0.03, 0, 0, 0), 5: (0.1, 0.2, 0, 0.001, 0.002), 6: (0.11, 0.21, 0.31, 0.0011, 0.0021)}
    rd = lambda a: np.array([float(f"{v:.12f}") for v in np.ravel(a)])
    for c, (img_id, cam_id, q, t, seen) in zip(cams, imgs):
        fx, fy, cx, cy = expK[cam_id]
        assert np.array_equal(c["K"], np.array([[fx, 0, cx], [0, fy, cy], [0, 0, 1.0]])) and c["has_K"]
        np.testing.assert_allclose(c["dist"], expD[cam_id], atol=1e-15)
        qq = rd(q); qq = qq / np.linalg.norm(qq); w, x, y, z = qq
        R = np.array([[1 - 2 * y * y - 2 * z * z, 2 * x * y - 2 * z * w, 2 * x * z + 2 * y * w], [2 * x * y + 2 * z * w, 1 - 2 * x * x - 2 * z * z, 2 * y * z - 2 * x * w],
                      [2 * x * z - 2 * y * w, 2 * y * z + 2 * x * w, 1 - 2 * x * x - 2 * y * y]])
        np.testing.assert_allclose(c["R"], R, atol=1e-14); np.testing.assert_allclose(c["t"], rd(t), atol=1e-15)
        np.testing.assert_allclose(c["C"], -R.T @ rd(t), atol=1e-13)
        assert c["wps"].tolist() == seen and c["name"] == f"im{img_id}.png"
        P = np.array([rd(pts[j]) if j != 7 else np.zeros(3) for j in seen])       # a point missing from points3D.txt stays at the origin
        dep = np.sort(np.array([np.float32(np.linalg.norm(c["C"] - p)) for p in P], np.float32))
        assert c["md"] == dep[len(dep) // 2]
    bad, err = _read_sfm_product(1, tmp_path / "nowhere")
    assert bad is None and "does not exist" in err
    (tmp_path / "cameras.txt").write_text("1 FISHEYE 10 10 1 2 3\n")
    bad, err = _read_sfm_product(1, tmp_path)
    assert bad is None and "FISHEYE unknown" in err



def test_cpp_frontend_compiles_against_the_public_headers(tmp_path):
    """the drop-in boundary is plain C++: examples/vsfm_frontend.cpp (the reference's main_vsfm.cpp flow on include/line3d.h +
    include/line3d_io.h) must compile warning-free with g++ alone, link against the in-tree library and - without a GPU - fail
    loudly instead of computing on the CPU"""
    from line3dpp_b200 import build
    so = build.build()
    exe = tmp_path / "vsfm_frontend"
    cmd = ["g++", "-std=c++17", "-Wall", "-Wextra", "-Werror", os.path.join(ROOT, "examples", "vsfm_frontend.cpp"), "-I" + os.path.join(ROOT, "include"),
           "-L" + os.path.dirname(so), "-ll3d_b200", "-Wl,-rpath," + os.path.dirname(so), "-o", str(exe)]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    nvm = tmp_path / "m.nvm"
    nvm.write_text("NVM_V3\n\n1\nimg0.jpg 1000 1 0 0 0 0 0 0 0 0\n\n1\n0 0 5 255 255 255 1 0 0 1.0 2.0\n")
    r = subprocess.run([str(exe), str(nvm), str(tmp_path), str(tmp_path)], capture_output=True, text=True)
    import torch
    if torch.cuda.is_available():
        assert r.returncode == 1 and "fewer than three usable images" in r.stderr, (r.returncode, r.stderr)
    else:
        assert r.returncode == 3 and "no usable CUDA device" in r.stderr, (r.returncode, r.stderr)



def test_reference_addimage_signature_compiles_against_eigen_opencv_headers(tmp_path):
    """include/line3d.h offers the reference's own addImage signature (line3D.h:104-108) when Eigen and OpenCV headers are on the
    include path.  Neither is installed here: compile against the stand-ins of oracle/ref_shim (the headers the verbatim reference
    build uses), link against the in-tree library and check that a view without segments is rejected, not detected on the CPU."""
    from line3dpp_b200 import build
    so = build.build()
    src = tmp_path / "facade.cpp"
    src.write_text(r"""
#include "line3d.h"
#ifndef L3DPP_WITH_EIGEN_OPENCV
#error "the Eigen / OpenCV overloads were not enabled"
#endif
#include <cstdio>
int main() {
    try {
        L3DPP::Line3D L("/tmp", true, -1, 3000, false, true);
        cv::Mat img(2304, 3072, CV_8U);
        Eigen::Matrix3d K = Eigen::Matrix3d::Identity(), R = Eigen::Matrix3d::Identity();
        Eigen::Vector3d t(0, 0, 1);
        std::list<unsigned int> nb; nb.push_back(1);
        std::vector<cv::Vec4f> segs(1, cv::Vec4f(1.f, 2.f, 300.f, 400.f));
        bool a = L.addImage(0u, img, K, R, t, 4.0f, nb, segs);
        bool b = L.addImage(1u, img, K, R, t, 4.0f, nb);          // no segments: rejected (no LSD here)
        std::printf("%d %d %zu\n", int(a), int(b), L.numImages());
        return (a && !b && L.numImages() == 1) ? 0 : 1;
    } catch (const std::exception& e) { std::printf("no GPU: %s\n", e.what()); return 3; }
}
""")
    exe = tmp_path / "facade"
    shim = os.path.join(ROOT, "oracle", "ref_shim")
    cmd = ["g++", "-std=c++17", "-Wall", "-Werror", str(src), "-I" + os.path.join(ROOT, "include"), "-I" + shim, "-L" + os.path.dirname(so), "-ll3d_b200",
           "-Wl,-rpath," + os.path.dirname(so), "-o", str(exe)]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    r = subprocess.run([str(exe)], capture_output=True, text=True)
    import torch
    assert r.returncode == (0 if torch.cuda.is_available() else 3), (r.returncode, r.stdout, r.stderr)


def test_no_cpu_fallback_without_gpu():
    """without a CUDA device the product must fail loudly, not compute on the CPU"""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    from line3dpp_b200 import capi, line3d
    h = ctypes.c_void_p()
    assert capi.lib().l3d_ctx_create(0, ctypes.byref(h)) < 0 and not h
    with pytest.raises(capi.L3DError):
        capi.Context(0)
    with pytest.raises(capi.L3DError):
        line3d.Line3D(False, True)


def test_product_never_imports_the_oracle():
    for root, _, files in os.walk(os.path.join(ROOT, "line3dpp_b200")):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".cc", ".h")):
                for line in open(os.path.join(root, f)):
                    if re.match(r"\s*(#\s*include|import|from)\b", line) or "CDLL" in line or "dlopen" in line:
                        assert "oracle" not in line, (f, line)


# ---------------------------------------------------------------------------------------------- BASELINE configs[0]: vsfm_result.nvm on the CPU path
def test_nvm_cpu_reference_run_matches_fixture_statistically(oracle):
    """testdata/vsfm_result.nvm, 26 views, default parameters (README.md:214-221), segments from cv2's LSD (committed
    inputs, tests/golden/make_nvm_inputs.py).  The oracle's restatement of the reference pipeline must reproduce the
    reference's own result testdata/Line3D++_ref statistically: line count within 3 %, symmetric chamfer distance of
    points sampled on the 3D segments below 0.5 % of the scene depth (median) - the same order as the distance between
    the oracle's REF_GPU and REF_CPU semantics.  Index parity is impossible here (different LSD build, SURVEY.md §4)."""
    from tests import nvm_util as nu
    oracle.set_threads(os.cpu_count() or 1)
    inp = nu.load_inputs()
    fx, fl, fr = nu.load_fixture()
    P = oracle.OraclePipeline(True, 1)
    nu.add_all(P.add_view, inp)
    assert P.match_images() == 0 and P.reconstruct(3, False) == 0
    oracle.set_threads(1)
    n_ref = len(set(fl.tolist()))
    assert abs(P.num_lines() - n_ref) <= 0.03 * n_ref, (P.num_lines(), n_ref)
    assert abs(len(P.residuals()) - len(fr)) <= 0.05 * len(fr)
    s = P.segments3d()
    mine = np.concatenate([s["p1"], s["p2"]], 1)
    a, b = nu.sample_points(mine), nu.sample_points(fx)
    depth = float(np.median(inp["median_depth"]))
    m1, p1 = nu.chamfer(a, b)
    m2, p2 = nu.chamfer(b, a)
    assert m1 < 0.005 * depth and m2 < 0.005 * depth, (m1, m2)
    assert p1 < 0.02 * depth and p2 < 0.02 * depth, (p1, p2)


def test_bench_helpers_without_gpu():
    """bench.py's bookkeeping helpers (committed ncu figures, nominal FP32 peak) never raise: a bad key or a CPU-only box yields None,
    and the committed capture of the dominant kernel is there for `roofline.traffic` / `roofline.executed`"""
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    b = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(b)
    cap = b.committed_capture("k_match_topk")
    assert cap and cap["warp_instructions"] > 1e10 and 0 < cap["issue_active_pct"] <= 100 and os.path.exists(os.path.join(ROOT, cap["capture"]))
    assert b.committed_traffic("k_match_topk") > 3e9
    assert b.committed_capture("no_such_kernel") is None and b.committed_traffic("no_such_kernel") is None
    assert b.nominal_fp32_tflops(None) is None
    v = b.nominal_fp32_tflops({"sm_mhz": 1965.0})        # None without a CUDA device, 148 x 128 x 2 x clock with one
    assert v is None or 50.0 < v < 100.0


def test_bench_dump_outputs_are_finite_floats(tmp_path):
    """bench.py --dump-outputs: float32 / float64 arrays only, every value finite (empty kNN slots hold -1, whatever the
    device left in them), the same seeded sample of view pairs every time"""
    import importlib.util
    from line3dpp_b200 import capi
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    b = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(b)
    rows, knn = 50, 10

    class FakeContext:        # the calls dump_outputs makes, with garbage (NaN / inf) in the slots past each row's count
        def match_counts(self):
            c = np.random.default_rng(1).integers(0, knn + 1, 6 * rows).astype(np.int32)
            return c, int(c.sum())

        def pair_row_offsets(self, n):
            return np.arange(n + 1, dtype=np.int64) * rows

        def pair_matches(self, p, ns):
            c = self.match_counts()[0][p * rows:(p + 1) * rows]
            r = np.zeros((ns, knn), capi.REC_DT)
            for f in ("overlap", "d_p1", "d_p2", "d_q1", "d_q2"):
                r[f] = np.where(np.arange(knn)[None] < c[:, None], 0.5 + p, np.nan if f == "overlap" else np.inf)
            r["tgt_seg"] = np.where(np.arange(knn)[None] < c[:, None], 7, 0xFFFFFFFF)
            return c, r

    class Scene:
        segs = [np.zeros((rows, 4), np.float32)] * 4
    pairs = np.array([[0, 1], [1, 2], [2, 3], [3, 0], [0, 2], [1, 3]], np.int32)
    for d in ("a", "b"):
        b.dump_outputs(FakeContext(), Scene(), pairs, str(tmp_path / d), nsample=3)
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == ["matches_per_pair.npy", "sample_counts.npy", "sample_depths.npy", "sample_overlap.npy", "sample_pairs.npy", "sample_tgt_seg.npy"]
    counts = np.load(tmp_path / "a" / "sample_counts.npy")
    for n in names:
        a = np.load(tmp_path / "a" / n)
        assert a.dtype in (np.float32, np.float64) and np.isfinite(a).all(), n
        assert np.array_equal(a, np.load(tmp_path / "b" / n)), n
    filled = np.arange(knn)[None, None] < counts[..., None]
    ov = np.load(tmp_path / "a" / "sample_overlap.npy")
    assert (ov[filled] > 0).all() and (ov[~filled] == -1).all() and (~filled).any()
    assert np.load(tmp_path / "a" / "matches_per_pair.npy").sum() == FakeContext().match_counts()[1]
