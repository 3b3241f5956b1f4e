"""The product (L3DPP::Line3D mirror on the B200) against the reference's WHOLE pipeline, UNMODIFIED: line3D.cc + view.cc +
cudawrapper.cu + sparsematrix.cc + clustering.cc compiled verbatim (oracle/_ref/libl3dref_full_gpu.so, nvcc -fmad=false, Eigen /
OpenCV / Boost replaced by the stand-ins of oracle/ref_shim) and run live on the same GPU through its own public calls
addImage / matchImages / reconstruct3Dlines.  No restated host logic is involved in these comparisons; what the reference
computed is recorded in tests/golden/ref_outputs_gpu_v1.npz (tests/golden/make_ref_outputs.py).

REF_GPU semantics: match ids, overlaps, depths and score3D bit-identical, list order identical, local ids / affinity edges
index-identical (weights: host libm vs libdevice, 1e-5 relative), 3D end points within 1e-6 scene units.
REF_CPU semantics (use_GPU=false) are checked against the golden vectors the verbatim CPU build produced
(tests/golden/ref_full_nvm_cpu_v1.npz)."""
import os

import numpy as np
import pytest

from line3dpp_b200 import line3d, synth
from tests import util
from tests.test_ref_full_cpu import digest_matches, G

pytestmark = pytest.mark.gpu

# weights: host libm vs libdevice; TOLERANCE on 3D end points: 1e-6 scene units
STAGE_TOL = {"est_p_smp": dict(rtol=0, atol=1e-12), "affraw_w_smp": dict(rtol=1e-5), "aff_w_smp": dict(rtol=1e-4, atol=1e-12),
             "seg_pts_smp": dict(rtol=0, atol=1e-6)}


@pytest.mark.parametrize("diffusion,collin,knn", [(False, -1.0, 10), (True, -1.0, 10), (True, 2.0, 10), (False, -1.0, 0)])
def test_synthetic_vs_reference_line3d_cc(ref, diffusion, collin, knn):
    sc = synth.make_scene(12, 600, 41, "ring3", collinear=collin > 0)
    L = line3d.Line3D(neighbors_by_worldpoints=False, use_gpu=True)
    L.add_scene(sc)
    L.match_images(knn=knn)
    L.reconstruct_3d_lines(3, diffusion, collin)
    r = ref(f"full/{diffusion}_{collin}_{knn}")
    util.check_record(util.product_record(L, sc.cam_ids, [len(s) for s in sc.segs], collin=collin > 0), r, STAGE_TOL)
    assert r["scored_n"].sum() > 20000 and r["aff_n"] > 3000 and r["num_lines"] > 150, (r["scored_n"].sum(), r["aff_n"], r["num_lines"])
    L.close()


def test_nvm_vs_reference_line3d_cc(ref, tmp_path):
    """BASELINE configs[1]: testdata/vsfm_result.nvm (26 views, neighbours from world points, default parameters) through the
    product on the B200 and through the unmodified reference's CUDA path on the same GPU: matches_, estimated_position3D_, A_,
    local ids, clusters and 3D segments index-exact; and the two text result files agree value by value."""
    from tests import nvm_util as nu
    inp = nu.load_inputs()
    L = line3d.Line3D(neighbors_by_worldpoints=True, use_gpu=True)
    nu.add_all(L.add_image, inp)
    L.match_images()
    L.reconstruct_3d_lines(3, False)
    nsegs = [len(s) for s in inp["segs"]]
    r = ref("full/nvm")
    mine = util.product_record(L, range(inp["V"]), nsegs)
    # result files: the reference's own writer vs the product's, same file name (createOutputFilename)
    L.save_txt(str(tmp_path))
    v = np.array(open(tmp_path / (str(r["txt_name"]) + ".txt")).read().split(), float)
    mine.update(txt_n=np.int64(len(v)), txt_smp=v[util.pick(len(v))], txt_name=r["txt_name"])
    util.check_record(mine, r, dict(STAGE_TOL, txt_smp=dict(rtol=1e-5, atol=1e-6)))
    assert r["scored_n"].sum() > 1000000 and r["num_lines"] > 2000, (r["scored_n"].sum(), r["num_lines"])
    # with diffusion on top (the reference supports re-running reconstruct3Dlines)
    L.reconstruct_3d_lines(3, True)
    util.check_record(util.product_record(L, range(inp["V"]), nsegs), ref("full/nvm_diffusion"), STAGE_TOL)
    L.close()


def test_nvm_refcpu_semantics_vs_verbatim_cpu_reference_golden():
    """use_GPU=false (the reference's CPU twins matchingCPU / scoringCPU, computed by the B200 in double) against the golden
    vectors of the verbatim CPU build on the nvm inputs.  The matching geometry is IEEE double add/mul/div/sqrt only: ids, overlaps
    and depths must be bit-identical wherever the match lists agree.  scoringCPU goes through expf/acosf (libdevice here, glibc in
    the golden), so a score that sits on a threshold (0.5 truncation, score > 0, 10 % of the best) can flip and, through the inverse
    matches, change the lists of later views: stated tolerance = at least 20 of 26 views with digest-identical scored lists,
    kept-match count within 0.5 %, line count within 1 %."""
    from tests import nvm_util as nu
    inp = nu.load_inputs()
    z = np.load(os.path.join(G, "ref_full_nvm_cpu_v1.npz"))
    L = line3d.Line3D(neighbors_by_worldpoints=True, use_gpu=False)
    nu.add_all(L.add_image, inp)
    L.match_images()
    assert np.array_equal(L.pairs(), z["pairs"])
    same = 0
    nk = 0
    for c in range(inp["V"]):
        m = L.view_matches(c, kept_only=False)
        same += int(len(m) == z["scored_count"][c] and np.array_equal(digest_matches(m), z["scored_sha"][c]))
        assert abs(len(m) - z["scored_count"][c]) <= 0.002 * z["scored_count"][c], c
        nk += len(L.view_matches(c, kept_only=True))
    print("REF_CPU on B200 vs verbatim CPU reference: digest-identical views", same, "of", inp["V"], "kept", nk, "vs", len(z["kept_src_cam"]))
    assert same >= 20
    assert abs(nk - len(z["kept_src_cam"])) <= 0.005 * len(z["kept_src_cam"])
    L.reconstruct_3d_lines(3, False)
    nl = L.stats()["lines3D"]
    assert abs(nl - 2428) <= 24, nl
    L.close()
