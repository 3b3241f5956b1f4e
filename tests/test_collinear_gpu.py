"""GPU parity of the collinearity row (SURVEY.md §8f-3): l3d_find_collinear against the UNMODIFIED reference kernel
(find_collinear_segments_GPU, oracle/_ref) and against the oracle's findCollinCPU restatement, and the collinearity
links of computingAffinityMatrix (line3D.cc:1904-1974) through the L3DPP::Line3D mirror against the oracle pipeline
driven by the reference kernels.  What the reference computed is recorded in tests/golden/ref_outputs_gpu_v1.npz
(tests/golden/make_ref_outputs.py)."""
import numpy as np
import pytest

from line3dpp_b200 import synth, line3d
from tests import util

pytestmark = pytest.mark.gpu


def _csr_to_dense(row_ptr, idx, n):
    Cm = np.zeros((n, n), np.uint8)
    for r in range(n):
        cols = idx[row_ptr[r]:row_ptr[r + 1]]
        assert np.all(np.diff(cols) > 0), "lists must be strictly ascending (collin_[i] order, view.cc:196-202)"
        Cm[r, cols] = 1
    return Cm


@pytest.fixture(scope="module")
def cscene():
    return util.collinear_scene()          # view 3 ragged + degenerate, view 4 a single segment, view 5 empty


@pytest.mark.parametrize("dist_t", [0.5, 2.0, 6.0])
def test_lists_equal_reference_kernel(gpu_ctx, cscene, ref, dist_t):
    gpu_ctx.set_views(util.scene_descs(cscene), cscene.segs)
    total = gpu_ctx.find_collinear(dist_t, 0)
    seen = 0
    for v, segs in enumerate(cscene.segs):
        rp, idx = gpu_ctx.collinear(v, len(segs))
        seen += len(idx)
        if len(segs) == 0:
            assert len(idx) == 0
            continue
        r = ref(f"collinear/{dist_t}")
        mine = _csr_to_dense(rp, idx, len(segs))
        assert util.sha(mine) == r[f"v{v}_sha"], f"view {v}: {mine.sum()} vs {r[f'v{v}_sum']} entries"
        if v == 0 and dist_t >= 2.0:
            assert r["v0_sum"] > 100          # the scene really has collinear fragments
    assert seen == total


@pytest.mark.parametrize("dist_t", [2.0, 6.0])
def test_refcpu_lists_equal_oracle_f64(gpu_ctx, cscene, oracle, dist_t):
    gpu_ctx.set_views(util.scene_descs(cscene), cscene.segs)
    gpu_ctx.find_collinear(dist_t, 1)
    for v, segs in enumerate(cscene.segs):
        if len(segs) == 0:
            continue
        rp, idx = gpu_ctx.collinear(v, len(segs))
        ref, _ = oracle.collinear(oracle.lib().orc_collinear_f64, segs, dist_t)
        assert np.array_equal(_csr_to_dense(rp, idx, len(segs)), ref), v


def test_oracle_f32_equals_reference_kernel(cscene, oracle, ref):
    for v in (0, 3):
        a, _ = oracle.collinear(oracle.lib().orc_collinear_f32, cscene.segs[v], 2.0)
        assert util.sha(a) == ref("collinear/2.0")[f"v{v}_sha"]


def test_switching_off_and_recompute(gpu_ctx, cscene):
    gpu_ctx.set_views(util.scene_descs(cscene), cscene.segs)
    n2 = gpu_ctx.find_collinear(2.0, 0)
    n6 = gpu_ctx.find_collinear(6.0, 0)
    assert n6 > n2 > 0
    assert gpu_ctx.find_collinear(0.0, 0) == 0
    assert gpu_ctx.find_collinear(2.0, 0) == n2


def _compare_reconstruction(L, P, atol):
    assert np.array_equal(L.local2global(), P.local2global())
    ei, ej, ew = L.affinity(raw=True)
    oi, oj, ow = P.affinity_raw()
    assert np.array_equal(ei, oi) and np.array_equal(ej, oj)
    np.testing.assert_allclose(ew, ow, rtol=1e-5)
    ei, ej, ew = L.affinity(raw=False)
    oi, oj, ow = P.affinity()
    assert np.array_equal(ei, oi) and np.array_equal(ej, oj)
    np.testing.assert_allclose(ew, ow, rtol=1e-4, atol=1e-12)
    assert L.stats()["lines3D"] == P.num_lines()
    mr, orr = L.residuals(), P.residuals()
    assert np.array_equal(mr["line"], orr["line"]) and np.array_equal(mr["cam"], orr["cam"]) and np.array_equal(mr["seg"], orr["seg"])
    ms, os_ = L.segments3d(), P.segments3d()
    assert np.array_equal(ms["line"], os_["line"])
    a = np.sort(np.stack([ms["p1"], ms["p2"]], 1), axis=1)
    b = np.sort(np.stack([os_["p1"], os_["p2"]], 1), axis=1)
    np.testing.assert_allclose(a, b, atol=atol)     # TOLERANCE on 3D endpoint positions: 1e-6 scene units


# affinity weights: host libm vs libdevice; TOLERANCE on 3D endpoint positions: 1e-6 scene units
RECON_TOL = {"affraw_w_smp": dict(rtol=1e-5), "aff_w_smp": dict(rtol=1e-4, atol=1e-12), "seg_pts_smp": dict(atol=1e-6)}


@pytest.mark.parametrize("diffusion,collin_t", [(False, 2.0), (True, 2.0), (True, 5.0)])
def test_collinearity_links_vs_reference_kernels(ref, diffusion, collin_t):
    sc = synth.make_scene(12, 500, 93, "ring3", collinear=True)
    L = line3d.Line3D(neighbors_by_worldpoints=False, use_gpu=True)
    L.add_scene(sc)
    L.match_images()
    L.reconstruct_3d_lines(3, diffusion, -1.0)
    base = L.stats()
    L.reconstruct_3d_lines(3, diffusion, collin_t)
    st = L.stats()
    # View::collin_ of every view, then the reconstruction
    util.check_record(util.product_record(L, sc.cam_ids, [len(s) for s in sc.segs], matching=False, collin=True), ref(f"collin_links/{diffusion}_{collin_t}"),
                      RECON_TOL)
    assert st["collinear_entries"] > 1000 and st["affinity_entries"] > base["affinity_entries"]    # the links are really there
    assert st["lines3D"] < base["lines3D"]                                                           # fragments were merged
    # switching the links off again reproduces the plain result
    L.reconstruct_3d_lines(3, diffusion, -1.0)
    again = L.stats()
    assert again["affinity_entries"] == base["affinity_entries"] and again["lines3D"] == base["lines3D"] and again["collinear_entries"] == 0
    L.close()


def test_collinearity_links_refcpu_vs_oracle(oracle):
    sc = synth.make_scene(10, 400, 94, "ring2", collinear=True)
    L = line3d.Line3D(neighbors_by_worldpoints=False, use_gpu=False)
    L.add_scene(sc)
    L.match_images()
    L.reconstruct_3d_lines(3, False, 2.0)
    P = oracle.OraclePipeline(False, False)
    P.add_scene(sc)
    P.match_images()
    assert P.reconstruct(3, False, 2.0) == 0
    assert L.stats()["collinear_entries"] > 500
    _compare_reconstruction(L, P, 1e-6)
    L.close()
