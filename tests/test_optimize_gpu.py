"""GPU parity of the line bundling (SURVEY.md §8f-4): l3d_optimize_lines against
  * the reference's OWN Ceres run: testdata/Line3D++_ref before / after result files (tests/golden/make_opt_fixture.py),
  * the oracle restatement of the same trust-region minimiser (same iterates, so agreement to rounding),
and the use_CERES flag of reconstruct3Dlines through the L3DPP::Line3D mirror against the oracle pipeline driven by the
reference kernels (recorded in tests/golden/ref_outputs_gpu_v1.npz by tests/golden/make_ref_outputs.py)."""
import numpy as np
import pytest

from line3dpp_b200 import synth, line3d
from tests import nvm_util as nu
from tests import util

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def pairs():
    before, after, ptr, res = nu.load_opt_pairs()
    cams, shift = nu.optimizer_inputs(nu.load_inputs())
    return dict(before=before + np.tile(shift, 2), after=after + np.tile(shift, 2), ptr=ptr, cam=res[:, 0].astype(np.int32), xy=res[:, 2:6], cams=cams)


def test_against_the_reference_ceres_result_files(gpu_ctx, pairs):
    out, valid, summ = gpu_ctx.optimize_lines(pairs["before"], pairs["ptr"], pairs["cam"], pairs["xy"], pairs["cams"], 250)
    assert valid.all() and summ[3] == 0 and summ[5] == len(out) and summ[7] > 10          # converged; kernels really ran
    assert summ[2] < 0.85 * summ[1]
    moved, gap = nu.line_gap(pairs["after"], pairs["before"]), nu.line_gap(pairs["after"], out)
    # fixture text rounding ~5e-6; the reference moved its lines by 3.8e-4 (median), up to 1.6e-2
    assert np.median(gap) < 2.5e-5 and np.percentile(gap, 90) < 1.5e-4 and np.percentile(gap, 99) < 8e-4, (np.median(gap), np.percentile(gap, [90, 99]))
    big = moved > 1e-3
    assert np.median(gap[big] / moved[big]) < 0.05


@pytest.mark.parametrize("max_iter", [250, 3, 0])
def test_same_iterates_as_the_oracle(gpu_ctx, oracle, pairs, max_iter):
    a, va, sa = gpu_ctx.optimize_lines(pairs["before"], pairs["ptr"], pairs["cam"], pairs["xy"], pairs["cams"], max_iter)
    b, vb, sb = oracle.optimize_lines(oracle.lib().orc_optimize_lines, pairs["before"], pairs["ptr"], pairs["cam"], pairs["xy"], pairs["cams"], max_iter)
    assert np.array_equal(va, vb)
    assert sa[0] == sb[0] and sa[3] == sb[3] and sa[4] == sb[4] and sa[5] == sb[5]         # iterations, termination, accepted steps, free lines
    np.testing.assert_allclose(sa[1:3], sb[1:3], rtol=1e-9)                                # initial / final cost
    # TOLERANCE on the optimised end points: 1e-8 scene units after a few iterations; at convergence a handful of lines with a
    # flat valley drift to ~2e-6 (device vs glibc exp/acos, amplified over ~30 iterations; Ceres stops on the TOTAL cost)
    np.testing.assert_allclose(a, b, atol=1e-8 if max_iter <= 3 else 1e-5)
    assert np.mean(np.abs(a - b) > 1e-8) < 0.03
    np.testing.assert_allclose(sa[6], sb[6], rtol=1e-2)     # trust-region radius (its update divides two nearly cancelling cost differences)


def test_subsets_ragged_and_degenerate_lines(gpu_ctx, oracle, pairs):
    sel = np.r_[0:40, 1000:1003]
    ptr = np.concatenate([[0], np.cumsum(np.diff(pairs["ptr"])[sel])])
    idx = np.concatenate([np.arange(pairs["ptr"][i], pairs["ptr"][i + 1]) for i in sel])
    p = pairs["before"][sel].copy()
    p[5, 2] = np.nan                                  # NaN Cayley coordinates -> the line is kept constant (optimization.cc:72-84) and dropped (293-298)
    ptr2 = np.concatenate([ptr, [ptr[-1]]])           # one more line without residuals
    p = np.concatenate([p, pairs["before"][7:8]])
    a, va, sa = gpu_ctx.optimize_lines(p, ptr2, pairs["cam"][idx], pairs["xy"][idx], pairs["cams"], 250)
    b, vb, sb = oracle.optimize_lines(oracle.lib().orc_optimize_lines, p, ptr2, pairs["cam"][idx], pairs["xy"][idx], pairs["cams"], 250)
    assert np.array_equal(va, vb) and va[5] == 0 and va[-1] == 1 and sa[5] == sb[5] == len(sel) - 1
    ok = va == 1
    np.testing.assert_allclose(a[ok], b[ok], atol=1e-5)
    e, ve, se = gpu_ctx.optimize_lines(np.zeros((0, 6)), [0], [], np.zeros((0, 4)), pairs["cams"], 10)
    assert len(e) == 0
    with pytest.raises(Exception):
        gpu_ctx.optimize_lines(p, ptr2, pairs["cam"][idx] + 1000, pairs["xy"][idx], pairs["cams"], 10)


@pytest.mark.parametrize("diffusion", [False, True])
def test_use_ceres_through_line3d_vs_oracle_pipeline(ref, diffusion):
    sc = synth.make_scene(12, 500, 96, "ring3", noise_px=1.0)
    L = line3d.Line3D(neighbors_by_worldpoints=False, use_gpu=True)
    L.add_scene(sc)
    L.match_images()
    L.reconstruct_3d_lines(3, diffusion, -1.0, False)
    plain = L.segments3d()
    L.reconstruct_3d_lines(3, diffusion, -1.0, True, 250)
    st = L.stats()
    r = ref(f"ceres/{diffusion}")
    sm = r["opt_summary"]
    assert st["opt_iterations"] == sm[0] and st["opt_iterations"] > 3
    np.testing.assert_allclose([st["opt_cost_before"], st["opt_cost_after"]], sm[1:3], rtol=1e-7)
    assert st["opt_cost_after"] < st["opt_cost_before"]
    ms = L.segments3d()
    mine = util.stage_record(num_lines=st["lines3D"], residuals=L.residuals(), segments=ms)
    keys = ("num_lines", "res_line_sha", "res_camseg_sha", "seg_n", "seg_pts_smp")
    util.check_record(mine, {k: r[k] for k in keys}, {"seg_pts_smp": dict(atol=1e-6)})     # TOLERANCE on 3D endpoint positions: 1e-6 scene units

    def gt(s):
        g = sc.lines3d; o = g[:, :3]; d = g[:, 3:] - o; d = d / np.linalg.norm(d, axis=1, keepdims=True)
        out = []
        for Pt in (s["p1"], s["p2"]):
            w = Pt[:, None, :] - o[None]
            out.append(np.linalg.norm(w - (w * d[None]).sum(-1, keepdims=True) * d[None], axis=-1).min(1))
        return np.concatenate(out).mean()
    assert gt(ms) < gt(plain)                        # the bundled lines are closer to the ground truth
    L.close()


def test_nvm_with_bundling_vs_optimized_fixture(ref):
    """testdata/vsfm_result.nvm with use_CERES on the B200 against the reference's OPTIMIZED result (statistical: the 2D
    segments of the fixture run are not reproducible, SURVEY.md §4) and against the oracle pipeline (1e-6)"""
    inp = nu.load_inputs()
    _, after, _, _ = nu.load_opt_pairs()
    L = line3d.Line3D(neighbors_by_worldpoints=True, use_gpu=True)
    nu.add_all(L.add_image, inp)
    L.match_images()
    L.reconstruct_3d_lines(3, False, -1.0, True, 250)
    r = ref("ceres/nvm")
    st = L.stats()
    assert st["lines3D"] == r["num_lines"] and st["opt_iterations"] == r["opt_summary"][0]
    ms = L.segments3d()
    util.check_record(util.stage_record(segments=ms), {k: r[k] for k in ("seg_n", "seg_pts_smp")}, {"seg_pts_smp": dict(atol=1e-6)})
    assert abs(st["lines3D"] - len(after)) <= 0.03 * len(after)
    mine = np.concatenate([ms["p1"], ms["p2"]], 1)
    depth = float(np.median(inp["median_depth"]))
    m1, _ = nu.chamfer(nu.sample_points(mine), nu.sample_points(after))
    m2, _ = nu.chamfer(nu.sample_points(after), nu.sample_points(mine))
    assert m1 < 0.005 * depth and m2 < 0.005 * depth, (m1, m2)
    L.close()
