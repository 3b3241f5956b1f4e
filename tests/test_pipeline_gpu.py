"""GPU parity of the full hot path (match -> orientation -> score -> inverse -> filter -> affinity -> diffusion ->
clusters -> 3D lines) through the L3DPP::Line3D mirror, against the oracle pipeline.

The oracle's host logic (oracle/l3d_oracle.cc) is driven twice:
  * with the UNMODIFIED reference kernels (oracle/_ref, -fmad=false) as its accelerator backend -> this IS the
    reference GPU path except for line3D.cc's host glue; the product must agree index-exactly and bit-exactly on
    overlaps / depths / scores;
  * with its CPU emulation, to show the same at libm tolerance.
What the reference kernels computed is recorded in tests/golden/ref_outputs_gpu_v1.npz (tests/golden/make_ref_outputs.py).
"""
import numpy as np
import pytest

from line3dpp_b200 import synth, line3d
from tests import util

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def scene():
    return synth.make_scene(14, 500, 31, "ring3")


@pytest.fixture(scope="module")
def product(scene):
    L = line3d.Line3D(neighbors_by_worldpoints=False, use_gpu=True)
    L.add_scene(scene)
    L.match_images()
    yield L
    L.close()


@pytest.fixture(scope="module")
def product_match(product, scene):
    return util.product_record(product, scene.cam_ids, None, recon=False)


@pytest.fixture(scope="module")
def oracle_cpu(scene, oracle):
    P = oracle.OraclePipeline(False, True)
    P.add_scene(scene)
    assert P.match_images() == 0
    return P


def test_view_pairs_and_regularisers(product_match, ref):
    r = ref("pipeline/match")
    assert product_match["pairs_sha"] == r["pairs_sha"]
    assert np.array_equal(product_match["view_info"], r["view_info"])


def test_scored_matches_bit_exact_vs_reference_kernels(product_match, ref):
    """all matches of every view right after scoring: order, ids, overlap, depths AND score3D bit-identical"""
    r = ref("pipeline/match")
    assert np.array_equal(product_match["scored_n"], r["scored_n"]) and product_match["scored_sha"] == r["scored_sha"]
    assert r["scored_n"].sum() > 20000


def test_kept_matches_and_estimates_vs_reference_kernels(product_match, ref):
    r = ref("pipeline/match")
    assert np.array_equal(product_match["kept_n"], r["kept_n"]) and product_match["kept_sha"] == r["kept_sha"]
    assert product_match["est_n"] == r["est_n"] and product_match["est_sha"] == r["est_sha"]
    np.testing.assert_allclose(product_match["est_p_smp"], r["est_p_smp"], rtol=0, atol=1e-12)
    assert r["est_n"] > 2000


def test_scored_matches_vs_cpu_oracle(product, oracle_cpu, scene):
    """same against the pure-CPU emulation: ids/overlap exact, depths/scores at libm tolerance (rsqrt/expf/acosf)"""
    nbad, noff, ntot = 0, 0, 0
    for cam in scene.cam_ids:
        mine = product.view_matches(cam, kept_only=False)
        ref = oracle_cpu.scored(cam)
        if len(mine) != len(ref) or not np.array_equal(mine["tgt_seg"], ref["tgt_seg"]):
            nbad += 1      # a depth sign / orientation / score>0 decision flipped by a 1-ulp libm difference: tolerated, counted
            continue
        assert np.array_equal(util.bits(mine["overlap"]), util.bits(ref["overlap"]))
        np.testing.assert_allclose(mine["d_p1"], ref["d_p1"], rtol=1e-3)
        # a similarity that sits at the 0.5 truncation (cudawrapper.cu:346) can flip with a 1-ulp expf difference and
        # moves the scores of that segment's matches by up to 0.5: allow a small fraction of outliers
        off = ~np.isclose(mine["score3D"], ref["score3D"], rtol=1e-3, atol=1e-4)
        noff += int(off.sum()); ntot += len(off)
        assert np.abs(mine["score3D"] - ref["score3D"])[off].max(initial=0) <= 1.0
    assert nbad <= 3 and ntot > 10000 and noff / ntot < 0.01


# affinity weights: host libm vs libdevice; TOLERANCE on 3D endpoint positions: 1e-6 scene units
RECON_TOL = {"affraw_w_smp": dict(rtol=1e-5), "aff_w_smp": dict(rtol=1e-4, atol=1e-12), "seg_pts_smp": dict(atol=1e-6)}


@pytest.mark.parametrize("diffusion", [False, True])
def test_reconstruction_vs_reference_kernels(scene, ref, diffusion):
    """affinity matrix before diffusion: same local ids, same edges in the same order, weights to libm tolerance; the matrix handed
    to the clustering (after diffusion if enabled); 3D lines (end points compared unordered: their order depends on the sign of
    the principal axis)"""
    L = line3d.Line3D(neighbors_by_worldpoints=False, use_gpu=True)
    L.add_scene(scene)
    L.match_images()
    L.reconstruct_3d_lines(3, diffusion)
    r = ref(f"pipeline/recon_{diffusion}")
    util.check_record(util.product_record(L, scene.cam_ids, None, matching=False), r, RECON_TOL)
    assert r["num_lines"] > 100
    L.close()


def test_rdd_bit_exact_vs_reference(gpu_ctx, oracle, ref):
    """l3d_rdd == verbatim SparseMatrix + replicator_dynamics_diffusion_GPU on a random symmetric affinity graph"""
    import ctypes as C
    ei, ej, ew, n = util.rdd_graph()
    r = ref("rdd")
    L = gpu_ctx.L
    oi, oj, ow = np.zeros_like(ei), np.zeros_like(ej), np.zeros_like(ew)
    ms = C.c_float(0)
    p = lambda x: x.ctypes.data_as(C.c_void_p)
    rc = L.l3d_rdd(gpu_ctx.h, n, C.c_longlong(len(ei)), p(ei), p(ej), p(ew), 10, p(oi), p(oj), p(ow), C.byref(ms))
    assert rc == 0
    assert util.sha(oi.astype(np.int64), oj.astype(np.int64)) == r["idx_sha"]
    assert util.sha(util.bits(ow)) == r["w_sha"]
    ci, cj, cw, _ = oracle.rdd(oracle.lib().orc_rdd_f32, ei, ej, ew, n)
    assert util.sha(ci.astype(np.int64), cj.astype(np.int64)) == r["idx_sha"] and util.sha(util.bits(cw)) == r["w_sha"]     # pins the CPU restatement too


# ---------------------------------------------------------------------------------------------- BASELINE configs[1]: vsfm_result.nvm on 1 x B200
def test_nvm_b200_vs_reference_kernels_and_fixture(ref):
    """testdata/vsfm_result.nvm through L3DPP::Line3D on the B200 (neighbours from world points, default parameters):
    index-exact against the oracle host logic driving the UNMODIFIED reference kernels, 3D endpoints within 1e-6 scene
    units, and statistically equal to the reference's own result fixture testdata/Line3D++_ref."""
    from tests import nvm_util as nu
    inp = nu.load_inputs()
    fx, fl, fr = nu.load_fixture()
    L = line3d.Line3D(neighbors_by_worldpoints=True, use_gpu=True)
    nu.add_all(L.add_image, inp)
    L.match_images()
    L.reconstruct_3d_lines(3, False)
    r = ref("pipeline/nvm")
    mine = util.product_record(L, range(inp["V"]), None)
    keys = ("pairs_sha", "kept_n", "kept_sha", "l2g_sha", "num_lines", "res_camseg_sha", "seg_n", "seg_pts_smp")
    util.check_record(mine, {k: r[k] for k in keys}, {"seg_pts_smp": dict(atol=1e-6)})
    st = L.stats()
    ms = L.segments3d()
    # statistical comparison with the reference's own output
    n_ref = len(set(fl.tolist()))
    assert abs(st["lines3D"] - n_ref) <= 0.03 * n_ref, (st["lines3D"], n_ref)
    mine = np.concatenate([ms["p1"], ms["p2"]], 1)
    depth = float(np.median(inp["median_depth"]))
    m1, _ = nu.chamfer(nu.sample_points(mine), nu.sample_points(fx))
    m2, _ = nu.chamfer(nu.sample_points(fx), nu.sample_points(mine))
    assert m1 < 0.005 * depth and m2 < 0.005 * depth, (m1, m2)
    print("nvm on B200:", st)
    import ctypes as C
    buf = C.create_string_buffer(512)
    assert L.L.l3dpp_output_filename(L.h, buf, 512) > 0
    assert buf.value.decode() == "Line3D++__W_FULL__N_10__sigmaP_2.5__sigmaA_10__epiOverlap_0.25__kNN_10__vis_3"      # the reference's own file name
    L.close()


def test_cluster_tail_reproduces_the_reference_result_file():
    """the host-side cluster -> 3D segment tail of the product (csrc/line3d_host.cc, findCollinearSegments line3D.cc:2342-2452)
    rebuilds every 3D segment of the reference's own result file from its lines + residuals"""
    import ctypes as C
    from tests import nvm_util as nu
    inp = nu.load_inputs()
    cam_segs, clusters = nu.fixture_clusters()
    L = line3d.Line3D(neighbors_by_worldpoints=True, use_gpu=True)
    for i in range(inp["V"]):
        w, h = inp["wh"][i]
        L.add_image(i, int(w), int(h), inp["K"][i], inp["R"][i], inp["t"][i], inp["median_depth"][i], inp["wps"][i], cam_segs[i])
    out = np.zeros((64, 6))
    p = lambda a: a.ctypes.data_as(C.c_void_p)

    def run(cl):
        n = L.L.l3dpp_collinear_from_cluster(L.h, p(np.ascontiguousarray(cl["p1p2"])), len(cl["cams"]), p(cl["cams"]), p(cl["segs"]), p(out), 64)
        return out[:n].copy()
    total, matched, extra, worst = nu.check_fixture_segments(run, clusters)
    assert total == 2501 and matched == total and worst < 5e-5, (total, matched, worst)
    assert extra <= 0.02 * total, extra
    L.close()


def test_writers_reproduce_the_reference_result_files_byte_for_byte(tmp_path):
    """save3DLinesAsTXT / saveResultAsOBJ / saveResultAsSTL (line3D.cc:2465-2687) against the reference's own files
    testdata/Line3D++_ref/*.{txt,obj,stl}: the lines parsed from those files are fed back into L3DPP::Line3D and the three
    writers must reproduce them byte for byte (SHA-256 committed by tests/golden/make_writer_golden.py); the file name of the
    nvm configuration is checked in test_nvm_b200_vs_reference_kernels_and_fixture"""
    import ctypes as C
    import hashlib
    import os
    from tests import nvm_util as nu
    inp = nu.load_inputs()
    segs3d, seg_line, res = nu.load_fixture()
    gold = np.load(os.path.join(nu.G, "ref_writers_v1.npz"))
    L = line3d.Line3D(neighbors_by_worldpoints=True, use_gpu=True)
    for i in range(inp["V"]):                           # views whose 2D segments sit at the reference's own segment ids
        r = res[res[:, 1] == i]
        lines = np.zeros((int(r[:, 2].max()) + 1 if len(r) else 1, 4), np.float32)
        lines[r[:, 2].astype(int)] = r[:, 3:7]
        w, h = inp["wh"][i]
        L.add_image(i, int(w), int(h), inp["K"][i], inp["R"][i], inp["t"][i], inp["median_depth"][i], inp["wps"][i], lines)
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    ids = sorted(set(seg_line.tolist()))
    nseg = np.array([(seg_line == ln).sum() for ln in ids], np.int32)
    nres = np.array([(res[:, 0] == ln).sum() for ln in ids], np.int32)
    order = np.argsort(res[:, 0], kind="stable")
    rc, rs = np.ascontiguousarray(res[order, 1], np.uint32), np.ascontiguousarray(res[order, 2], np.uint32)

    def written(segs, save, ext):
        assert L.L.l3dpp_set_lines(L.h, len(ids), p(nseg), p(np.ascontiguousarray(segs, np.float64)), p(nres), p(rc), p(rs)) == 0
        d = tmp_path / ext
        d.mkdir()
        assert save(L.h, str(d).encode()) == 0
        files = os.listdir(d)
        assert len(files) == 1 and files[0].endswith("." + ext)
        return hashlib.sha256(open(d / files[0], "rb").read()).hexdigest()
    assert len(gold["stl_segs"]) == len(segs3d) == nseg.sum()
    assert written(segs3d, L.L.l3dpp_save_txt, "txt") == str(gold["sha_txt"])
    assert written(segs3d, L.L.l3dpp_save_obj, "obj") == str(gold["sha_obj"])
    assert written(gold["stl_segs"], L.L.l3dpp_save_stl, "stl") == str(gold["sha_stl"])
    L.close()


def test_add_image_and_writer_errors_are_reported(tmp_path):
    """ADVICE r1: addImage failures are attributable (status + sticky lastError), writers report unwritable folders"""
    sc = synth.make_scene(6, 200, 3, "ring2")
    L = line3d.Line3D(neighbors_by_worldpoints=False, use_gpu=True)
    L.add_scene(sc)
    import ctypes as C
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    K, R, t = np.ascontiguousarray(sc.K[0]), np.ascontiguousarray(sc.R[0]), np.ascontiguousarray(sc.t[0])
    nb, sg = np.ascontiguousarray(sc.neighbors[0], np.uint32), np.ascontiguousarray(sc.segs[0], np.float32)
    add = lambda cam, w: L.L.l3dpp_add_image(L.h, C.c_uint(cam), w, w * 3 // 4, p(K), p(R), p(t), C.c_float(4.0), p(nb), len(nb), p(sg), len(sg))
    assert add(0, 3072) < 0 and b"already in use" in L.L.l3dpp_last_error(L.h)          # duplicate camera id
    assert add(77, 100) < 0 and b"too small" in L.L.l3dpp_last_error(L.h)
    assert add(78, 3072) == 0                                                          # a success ...
    assert b"too small" in L.L.l3dpp_last_error(L.h)                                   # ... does not wipe the earlier failure
    L.match_images()
    L.reconstruct_3d_lines(3, False)
    assert L.stats()["lines3D"] > 20
    with pytest.raises(Exception) as e:
        L.save_txt(str(tmp_path / "does" / "not" / "exist"))
    assert "cannot open" in str(e.value)
    L.save_txt(str(tmp_path))
    assert any(f.name.endswith(".txt") for f in tmp_path.iterdir())
    L.close()
