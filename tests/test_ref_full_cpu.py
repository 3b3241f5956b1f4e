"""The oracle's restatement of the reference's HOST logic (oracle/l3d_oracle.cc: Line3D / View, line3D.cc + view.cc) pinned
index-exactly on the UNMODIFIED reference: line3D.cc + view.cc + clustering.cc compiled verbatim from /root/reference
against the Eigen/OpenCV/Boost stand-ins of oracle/ref_shim (oracle/_ref/libl3dref_full_cpu.so, oracle/Makefile), CPU code
path, single-threaded.

  * on small synthetic scenes (explicit neighbours, collinearity links, keep-all kNN), through
    tests/golden/ref_outputs_cpu_v1.npz, which that library produced (tests/golden/make_ref_outputs.py);
  * through tests/golden/ref_full_nvm_cpu_v1.npz, which the same library produced on the committed vsfm_result.nvm inputs
    (26 views, neighbours from world points, default parameters; tests/golden/make_ref_full_golden.py).
"""
import hashlib
import os

import numpy as np
import pytest

from line3dpp_b200 import synth
from tests import util

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
IDS = ("src_cam", "src_seg", "tgt_cam", "tgt_seg")
GEO = ("overlap", "d_p1", "d_p2", "d_q1", "d_q2")


@pytest.mark.parametrize("V,N,nb,collin,knn", [(8, 300, "ring2", -1.0, 10), (10, 250, "ring3", 2.0, 10), (6, 200, "ring2", -1.0, 0)])
def test_oracle_host_logic_vs_verbatim_line3d_cc(oracle, tmp_path, V, N, nb, collin, knn):
    """every stage of the reference pipeline, verbatim (recorded in tests/golden/ref_outputs_cpu_v1.npz) vs restated: matches
    after scoring, kept matches, regularisers, best estimates, collinear lists, local ids, affinity edges, clusters' residuals
    and 3D segments, and the text result file.  Ids, overlaps and depths bit-identical; score3D within a few ulps (libm
    expf/acosf are called through different expression types by the two builds)"""
    sc = synth.make_scene(V, N, 7, nb, collinear=collin > 0)
    O = oracle.OraclePipeline(False, 0)
    O.add_scene(sc)
    O.match_images(knn=knn)
    O.reconstruct(3, False, collin)
    mine = util.dump_record(O, sc.cam_ids, [len(s) for s in sc.segs], collin=collin > 0, exact_scores=False)
    O.save_txt(str(tmp_path / "oracle.txt"))
    v = np.array(open(tmp_path / "oracle.txt").read().split(), float)
    mine.update(txt_n=np.int64(len(v)), txt_smp=v[util.pick(len(v))])
    ref = util.load_record(np.load(os.path.join(G, "ref_outputs_cpu_v1.npz")), f"host_logic/{V}_{N}_{nb}_{collin}_{knn}")
    ulps = dict(rtol=4.8e-7, atol=0)
    util.check_record(mine, ref, {"scored_score_smp": ulps, "kept_score_smp": ulps, "est_score_smp": ulps, "est_p_smp": dict(rtol=0, atol=1e-13),
                                  "affraw_w_smp": dict(rtol=1e-6), "seg_pts_smp": dict(rtol=0, atol=1e-12), "txt_smp": dict(rtol=1e-5, atol=1e-9)},
                      skip=("aff_n", "aff_idx_sha", "aff_w_smp"))
    assert ref["affraw_n"] > 1000 and ref["num_lines"] > 50


def digest_matches(m):
    h = hashlib.sha256()
    for f in IDS + GEO:
        h.update(np.ascontiguousarray(m[f]).tobytes())
    return np.frombuffer(h.digest(), np.uint8)


def check_against_nvm_golden(pipe, V, scored, kept, exact_geo=True):
    """pipe: anything with the OraclePipeline dump interface that has run the nvm inputs with REF_CPU semantics"""
    z = np.load(os.path.join(G, "ref_full_nvm_cpu_v1.npz"))
    assert np.array_equal(pipe.pairs(), z["pairs"])
    for c in range(V):
        m = scored(c)
        assert len(m) == z["scored_count"][c], (c, len(m), z["scored_count"][c])
        if exact_geo:
            assert np.array_equal(digest_matches(m), z["scored_sha"][c]), c
        assert abs(float(m["score3D"].astype(np.float64).sum()) - z["scored_score_sum"][c]) <= 1e-4 * max(1.0, z["scored_score_sum"][c])
        k, md = pipe.view_info(c)
        assert np.float32(k) == z["view_info"][c, 0] and np.float32(md) == z["view_info"][c, 1], c
    k = np.concatenate([kept(c) for c in range(V)])
    assert len(k) == len(z["kept_src_cam"])
    for f in IDS:
        assert np.array_equal(k[f], z["kept_" + f]), f
    if exact_geo:
        assert np.array_equal(digest_matches(k), z["kept_sha"])
    np.testing.assert_allclose(k["score3D"], z["kept_score3D"], rtol=2e-5, atol=1e-6)
    best, P = pipe.estimates()
    assert np.array_equal(np.stack([best[f] for f in IDS], 1), z["est_src"])
    np.testing.assert_allclose(P, z["est_P"], rtol=0, atol=1e-12)


def check_reconstruction_against_nvm_golden(local2global, affinity_raw, segments3d, residuals):
    z = np.load(os.path.join(G, "ref_full_nvm_cpu_v1.npz"))
    assert np.array_equal(local2global, z["l2g"])
    ei, ej, ew = affinity_raw
    assert np.array_equal(ei, z["aff_i"]) and np.array_equal(ej, z["aff_j"])
    np.testing.assert_allclose(ew, z["aff_w"], rtol=1e-5)
    r = residuals
    assert np.array_equal(np.stack([r["line"], r["cam"].astype(np.int32), r["seg"].astype(np.int32)], 1), z["res"])
    s = segments3d
    assert np.array_equal(s["line"], z["seg_line"])
    a = np.sort(np.stack([s["p1"], s["p2"]], 1), axis=1)
    b = np.sort(z["seg_p1p2"].reshape(-1, 2, 3), axis=1)
    np.testing.assert_allclose(a, b, rtol=0, atol=1e-6)      # TOLERANCE on 3D end points: 1e-6 scene units
    return len(s), len(set(s["line"].tolist()))


def test_oracle_vs_verbatim_reference_on_nvm_and_fixture(oracle, tmp_path):
    """BASELINE configs[0]: testdata/vsfm_result.nvm, 26 views, CPU path, default parameters (README.md:214-221) on the
    committed cv2-LSD segments.  (1) The oracle's restatement reproduces the VERBATIM reference pipeline's result on these
    inputs index-exactly at every stage (golden made by tests/golden/make_ref_full_golden.py).  (2) Both agree with the
    reference's own shipped result testdata/Line3D++_ref statistically - its input segments came from another LSD build
    (SURVEY.md §4), so segment ids cannot line up: line count within 3 %, symmetric chamfer distance below 0.5 % of the
    scene depth."""
    from tests import nvm_util as nu
    oracle.set_threads(os.cpu_count() or 1)
    inp = nu.load_inputs()
    P = oracle.OraclePipeline(True, 0)
    nu.add_all(P.add_view, inp)
    assert P.match_images() == 0 and P.reconstruct(3, False) == 0
    oracle.set_threads(1)
    check_against_nvm_golden(P, inp["V"], P.scored, P.matches)
    nseg, nlines = check_reconstruction_against_nvm_golden(P.local2global(), P.affinity_raw(), P.segments3d(), P.residuals())
    assert (nlines, nseg) == (2428, 2440)
    # the reference's own text writer produced this file from the same run
    z = np.load(os.path.join(G, "ref_full_nvm_cpu_v1.npz"))
    assert str(z["txt_name"]) == "Line3D++__W_FULL__N_10__sigmaP_2.5__sigmaA_10__epiOverlap_0.25__kNN_10__vis_3"
    # (2) statistics against testdata/Line3D++_ref
    fx, fl, fr = nu.load_fixture()
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
