"""GPU parity of the matching kernels against the UNMODIFIED reference kernels (oracle/_ref, built with -fmad=false; their
outputs recorded in tests/golden/ref_outputs_gpu_v1.npz by tests/golden/make_ref_outputs.py) and the CPU oracle.  Everything
goes through the C ABI (line3dpp_b200.capi -> libl3d_b200.so)."""
import numpy as np
import pytest

from line3dpp_b200 import synth
from tests import util

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def scene():
    return synth.make_scene(8, 700, 11, "dense")


@pytest.fixture(scope="module")
def loaded(gpu_ctx, scene):
    gpu_ctx.set_views(util.scene_descs(scene), scene.segs)
    return gpu_ctx


PAIRS = [(0, 1), (0, 4), (2, 3), (5, 1), (7, 6)]


def check_lists(counts, recs, r, max_ties=None, what=""):
    """kNN lists against the recorded reference: same counts, same sets up to exact ties at the k-th place, and (max_ties)
    at most that many rows whose sets differ at all"""
    assert np.array_equal(counts, r["counts"]), (what, np.flatnonzero(counts != r["counts"])[:10])
    assert util.tie_sha(counts, recs) == r["tie_sha"], what
    if max_ties is not None:
        assert (util.row_shas(counts, recs) != r["row_sha"]).sum() <= max_ties, what
    for row in range(len(counts)):
        ov = recs[row, :counts[row]]["overlap"]
        assert np.all(ov[:-1] >= ov[1:])


@pytest.mark.parametrize("src,tgt", PAIRS)
def test_dense_bit_exact_vs_reference_kernel(loaded, scene, ref, src, tgt):
    """l3d_match_dense == verbatim K_match_lines (cudawrapper.cu:186-253), every cell, every bit."""
    pi = util.pair_inputs(scene, src, tgt)
    r = ref(f"dense/{src}_{tgt}")
    dep, ov = loaded.match_dense(src, tgt, pi["F"], 0.25, len(pi["ls"]), len(pi["lt"]))
    assert util.sha(util.bits(ov)) == r["ov_sha"]
    assert util.sha(util.bits(dep)) == r["dep_sha"]
    # the conservative pre-filter must never change a result
    dep2, ov2 = loaded.match_dense(src, tgt, pi["F"], 0.25, len(pi["ls"]), len(pi["lt"]), nofilter=True)
    assert util.sha(util.bits(ov2)) == r["ov_sha"] and util.sha(util.bits(dep2)) == r["dep_sha"]
    assert r["nsel"] > 100   # the case is not vacuous


@pytest.mark.parametrize("src,tgt", PAIRS[:3])
def test_dense_cpu_oracle_matches_reference(scene, oracle, ref, src, tgt):
    """pins the CPU restatement: overlap bit-exact, depths to 1e-5 relative (host rsqrt differs from MUFU.RSQ) on a seeded
    sample of the cells above the threshold."""
    pi = util.pair_inputs(scene, src, tgt)
    r = ref(f"dense/{src}_{tgt}")
    odep, oov, _ = oracle.match_dense(oracle.lib().orc_match_dense_f32, pi["ls"], pi["lt"], pi["F"], pi["Rs"], pi["Rt"], pi["Cs"], pi["Ct"], 0.25)
    assert util.sha(util.bits(oov)) == r["ov_sha"]
    sel = np.flatnonzero(oov.reshape(-1) > 0.25)
    assert len(sel) == r["nsel"] and np.array_equal(sel[util.pick(len(sel))], r["cells"])
    odep, rdep = odep.reshape(-1, 4)[r["cells"]], r["dep"]
    rel = np.abs(odep - rdep) / np.maximum(np.abs(rdep), 1e-3)
    assert np.median(rel) < 1e-6 and np.quantile(rel, 0.999) < 1e-2     # ill-conditioned depths (n.ray ~ 0) amplify the rsqrt difference
    assert np.array_equal(np.sign(odep), np.sign(rdep)) or (np.sign(odep) != np.sign(rdep)).mean() < 1e-5


def test_topk_vs_reference_wrapper(loaded, scene, ref):
    """l3d_match_pairs == verbatim match_lines_GPU (kernel + D2H + host priority queue, cudawrapper.cu:549-658):
    same match set per source segment, bit-exact payload.  Order inside a row: overlap descending.  The only acceptable
    difference is a tie in overlap at the k-th place (std::priority_queue order is unspecified), in at most 2 rows."""
    pairs = np.array(PAIRS, np.int32)
    loaded.match_pairs(pairs, util.pair_F(scene, pairs), 0.25, 10)
    for p, (src, tgt) in enumerate(PAIRS):
        counts, recs = loaded.pair_matches(p, len(scene.segs[src]))
        check_lists(counts, recs, ref(f"topk/{src}_{tgt}"), max_ties=2, what=(src, tgt))
        assert counts.sum() > 1000


@pytest.mark.parametrize("f64", [False, True])
def test_keep_all_matches(loaded, scene, oracle, ref, f64):
    """kNN <= 0: every cell with overlap > epi and positive depths is kept, in ascending target order
    (cudawrapper.cu:628-636 / line3D.cc:988-996) -- against the verbatim wrapper (float) and the oracle's matchingCPU (double)"""
    pairs = np.array(PAIRS[:3], np.int32)
    if f64:
        Fd = np.stack([synth.fundamental(scene.K[s], scene.R[s], scene.t[s], scene.K[t], scene.R[t], scene.t[t]).reshape(9) for s, t in pairs])
        loaded.match_pairs_f64(pairs, Fd, 0.25, 0)
    else:
        loaded.match_pairs(pairs, util.pair_F(scene, pairs), 0.25, -1)
    stride = loaded.L.l3d_match_stride(loaded.h)
    assert stride > 10
    biggest = 0
    for p, (src, tgt) in enumerate(pairs):
        pi = util.pair_inputs(scene, src, tgt)
        if f64:
            RtKinv, C = synth.camera_blocks(scene)
            rcounts, rout, rtotal, _ = oracle.match_lines(oracle.lib().orc_match_lines_f64, pi["ls"], pi["lt"], Fd[p], RtKinv[src].reshape(9),
                                                          RtKinv[tgt].reshape(9), C[src], C[tgt], src, tgt, 0.25, 0, f64=True)
        counts, recs = loaded.pair_matches(p, len(pi["ls"]))
        biggest = max(biggest, int(counts.max()))
        if not f64:
            assert util.list_sha(counts, recs) == ref(f"keep_all/{src}_{tgt}")["list_sha"], (src, tgt)    # same members, same ORDER, bit-exact payload
            continue
        assert np.array_equal(counts, rcounts) and rtotal == counts.sum()
        for r in range(len(counts)):
            a, b = recs[r, :counts[r]], rout[r, :counts[r]]
            for f in ("tgt_seg", "overlap", "d_p1", "d_p2", "d_q1", "d_q2"):
                assert a[f].tobytes() == b[f].tobytes(), (src, tgt, r, f)          # same members, same ORDER, bit-exact payload
    assert biggest <= stride


def test_keep_all_pipeline_vs_reference_kernels(ref):
    """matchImages(kNN = -1) end to end: scored matches bit-identical to the reference kernels behind the oracle host logic"""
    from line3dpp_b200 import line3d
    sc = synth.make_scene(6, 250, 13, "ring2")
    L = line3d.Line3D(neighbors_by_worldpoints=False)
    L.add_scene(sc); L.match_images(knn=-1)
    r = ref("keep_all_pipeline")
    mine = util.stage_record(scored=[L.view_matches(cam, False) for cam in sc.cam_ids])
    assert np.array_equal(mine["scored_n"], r["scored_n"]) and mine["scored_sha"] == r["scored_sha"]
    assert r["scored_n"].sum() > 3000
    L.reconstruct_3d_lines(3, False)
    assert L.stats()["lines3D"] == r["num_lines"] > 20
    L.close()


@pytest.mark.parametrize("chunks", [1, 5, 64])
def test_match_pairs_host_equals_match_then_download(loaded, scene, chunks):
    """l3d_match_pairs_host (chunked launches + overlapped D2H) delivers exactly what l3d_match_pairs + download delivers"""
    import torch
    from line3dpp_b200 import capi
    pairs = synth.view_pairs(scene.neighbors)[:9]
    F = util.pair_F(scene, pairs)
    loaded.match_pairs(pairs, F, 0.25, 10)
    want_counts, total = loaded.match_counts()
    want = [loaded.pair_matches(p, len(scene.segs[s])) for p, (s, t) in enumerate(pairs)]
    rows = loaded.match_total_rows()
    counts = torch.full((rows,), -7, dtype=torch.int32).pin_memory()
    recs = torch.zeros(rows * 10 * 24, dtype=torch.uint8).pin_memory()
    loaded.match_pairs_host(pairs, F, counts.data_ptr(), recs.data_ptr(), 0.25, 10, chunks)
    loaded.sync()
    assert np.array_equal(counts.numpy(), want_counts) and total > 5000
    got = recs.numpy().view(capi.REC_DT).reshape(rows, 10)
    off = loaded.pair_row_offsets(len(pairs))
    for p in range(len(pairs)):
        c, r = want[p]
        for i in range(len(c)):
            assert got[off[p] + i, :c[i]].tobytes() == r[i, :c[i]].tobytes()
    # the device-side result is the same object the sweep would consume
    again, _ = loaded.match_counts()
    assert np.array_equal(again, want_counts)


def test_topk_matches_csr_and_counts(loaded, scene):
    pairs = np.array(PAIRS, np.int32)
    loaded.match_pairs(pairs, util.pair_F(scene, pairs), 0.25, 10)
    counts, total = loaded.match_counts()
    row_ptr, recs = loaded.matches_csr()
    assert row_ptr[-1] == total == len(recs)
    assert np.array_equal(np.diff(row_ptr), counts)
    off = 0
    for p, (src, tgt) in enumerate(PAIRS):
        c, r = loaded.pair_matches(p, len(scene.segs[src]))
        for row in (0, 17, len(c) - 1):
            a = recs[row_ptr[off + row]:row_ptr[off + row + 1]]
            assert np.array_equal(a, r[row, :c[row]])
        off += len(c)


@pytest.mark.parametrize("knn", [1, 3, 32])
def test_topk_other_k(loaded, scene, oracle, knn):
    """k other than the default, against the CPU oracle (overlap + membership are bitwise reproducible on the CPU)."""
    pairs = np.array([(1, 2)], np.int32)
    loaded.match_pairs(pairs, util.pair_F(scene, pairs), 0.3, knn)
    pi = util.pair_inputs(scene, 1, 2)
    ocounts, oout, _, _ = oracle.match_lines(oracle.lib().orc_match_lines_f32, pi["ls"], pi["lt"], pi["F"], pi["Rs"], pi["Rt"], pi["Cs"], pi["Ct"], 1, 2, 0.3, knn)
    counts, recs = loaded.pair_matches(0, len(pi["ls"]))
    assert np.array_equal(counts, ocounts)
    f = ("tgt_seg", "overlap")
    assert util.rows_as_sets(counts, recs, f) == util.rows_as_sets(ocounts, oout, f)


def test_ragged_and_tiny_views(gpu_ctx, oracle):
    """views of different sizes incl. 1 segment, sizes not multiples of any tile; the overflow/prune path (every
    target segment identical -> >64 survivors per row)."""
    sc = synth.make_scene(4, 333, 5, "dense")
    sc.segs[1] = sc.segs[1][:1].copy()
    sc.segs[2] = sc.segs[2][:65].copy()
    # view 3: 200 copies of a segment that matches view 0's segment 0 -> forces list overflow + ties
    pi = util.pair_inputs(sc, 0, 3)
    c, o, _, _ = oracle.match_lines(oracle.lib().orc_match_lines_f32, pi["ls"], pi["lt"], pi["F"], pi["Rs"], pi["Rt"], pi["Cs"], pi["Ct"], 0, 3, 0.25, 10)
    r = int(np.argmax(c))
    sc.segs[3] = np.repeat(sc.segs[3][o[r, 0]["tgt_seg"]][None], 200, axis=0).copy()
    gpu_ctx.set_views(util.scene_descs(sc), sc.segs)
    pairs = np.array([(0, 1), (1, 0), (0, 2), (2, 1), (0, 3), (3, 2)], np.int32)
    gpu_ctx.match_pairs(pairs, util.pair_F(sc, pairs), 0.25, 10)
    for p, (s, t) in enumerate(pairs):
        pi = util.pair_inputs(sc, s, t)
        oc, oo, _, _ = oracle.match_lines(oracle.lib().orc_match_lines_f32, pi["ls"], pi["lt"], pi["F"], pi["Rs"], pi["Rt"], pi["Cs"], pi["Ct"], s, t, 0.25, 10)
        counts, recs = gpu_ctx.pair_matches(p, len(pi["ls"]))
        assert np.array_equal(counts, oc), (s, t)
        if t == 3:   # all ties: ours must be the 10 smallest tgt indices
            rr = np.flatnonzero(counts == 10)
            assert len(rr) > 0
            for row in rr:
                assert list(recs[row]["tgt_seg"]) == list(range(10))
        else:
            f = ("tgt_seg", "overlap")
            assert util.rows_as_sets(counts, recs, f) == util.rows_as_sets(oc, oo, f)


def test_filter_never_drops_at_scale(gpu_ctx, oracle):
    """2000x2000 pairs from several geometries: filtered dense kernel == unfiltered dense kernel, all cells."""
    sc = synth.make_scene(6, 2000, 21, "dense")
    gpu_ctx.set_views(util.scene_descs(sc), sc.segs)
    for (s, t) in [(0, 1), (0, 3), (2, 5), (4, 1)]:
        F = util.pair_F(sc, [(s, t)])[0]
        d1, o1 = gpu_ctx.match_dense(s, t, F, 0.25, 2000, 2000)
        d2, o2 = gpu_ctx.match_dense(s, t, F, 0.25, 2000, 2000, nofilter=True)
        assert np.array_equal(util.bits(o1), util.bits(o2))
        assert np.array_equal(util.bits(d1), util.bits(d2))


def test_sharded_matching_equals_unsharded(gpu_ctx):
    """pair sharding (what N ranks do) does not change a single bit: match the full pair list at once, then the two
    rank shards separately, and compare every record."""
    from line3dpp_b200 import shard
    sc = synth.make_scene(12, 300, 13, "ring3")
    gpu_ctx.set_views(util.scene_descs(sc), sc.segs)
    pairs = synth.view_pairs(sc.neighbors)
    F = util.pair_F(sc, pairs)
    gpu_ctx.match_pairs(pairs, F, 0.25, 10)
    row_ptr, recs = gpu_ctx.matches_csr()
    full = {}
    off = 0
    for p, (s, t) in enumerate(pairs):
        n = len(sc.segs[s])
        full[(int(s), int(t))] = (np.diff(row_ptr[off:off + n + 1]).copy(), recs[row_ptr[off]:row_ptr[off + n]].copy())
        off += n
    seen = 0
    for rank in range(2):
        mine = shard.rank_pairs(pairs, rank, 2, sc.num_views)
        sel = np.array([i for i, pr in enumerate(pairs.tolist()) if pr in mine.tolist()])
        gpu_ctx.match_pairs(mine, F[sel], 0.25, 10)
        rp, rc = gpu_ctx.matches_csr()
        off = 0
        for (s, t) in mine:
            n = len(sc.segs[s])
            cnt, rr = full[(int(s), int(t))]
            assert np.array_equal(np.diff(rp[off:off + n + 1]), cnt)
            assert np.array_equal(rc[rp[off]:rp[off + n]], rr)
            off += n
            seen += 1
    assert seen == len(pairs)


def test_large_target_views_reuse_the_tma_ring(gpu_ctx, oracle):
    """target views larger than the resident TMA ring (3 x 1024 segments): stages are refilled, last stage partial"""
    sc = synth.make_scene(3, 3600, 17, "dense")
    sc.segs[0] = sc.segs[0][:150].copy()
    sc.segs[2] = np.concatenate([sc.segs[2], sc.segs[1][:3409]]).copy()      # 7009 segments: 7 stages, 865 in the last
    gpu_ctx.set_views(util.scene_descs(sc), sc.segs)
    pairs = np.array([(0, 1), (0, 2)], np.int32)
    gpu_ctx.match_pairs(pairs, util.pair_F(sc, pairs), 0.25, 10)
    for p, (s, t) in enumerate(pairs):
        pi = util.pair_inputs(sc, s, t)
        oc, oo, _, _ = oracle.match_lines(oracle.lib().orc_match_lines_f32, pi["ls"], pi["lt"], pi["F"], pi["Rs"], pi["Rt"], pi["Cs"], pi["Ct"], s, t, 0.25, 10)
        counts, recs = gpu_ctx.pair_matches(p, len(pi["ls"]))
        assert np.array_equal(counts, oc)
        f = ("tgt_seg", "overlap")
        assert util.rows_as_sets(counts, recs, f) == util.rows_as_sets(oc, oo, f)


def test_capi_error_behaviour(gpu_ctx):
    """every entry returns a negative l3d_status + message instead of printing and carrying on (dataArray.h:198-237)"""
    import ctypes as C
    from line3dpp_b200 import capi
    L = gpu_ctx.L
    fresh = capi.Context(0)
    assert L.l3d_match_pairs(fresh.h, 0, None, None, C.c_float(0.25), 10) == -3            # L3D_ERR_STATE: no views yet
    assert b"l3d_set_views" in L.l3d_last_error(fresh.h)
    assert L.l3d_score_sweep(fresh.h, C.c_float(200), C.c_float(.5), C.c_float(.75), C.c_float(.1)) == -3
    sc = synth.make_scene(3, 50, 2, "dense")
    fresh.set_views(util.scene_descs(sc), sc.segs)
    pairs = np.array([[0, 7]], np.int32)
    F = np.zeros((1, 9), np.float32)
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    assert L.l3d_match_pairs(fresh.h, 1, p(pairs), p(F), C.c_float(0.25), 10) == -1         # view index out of range
    pairs[0, 1] = 1
    assert L.l3d_match_pairs(fresh.h, 1, p(pairs), p(F), C.c_float(0.25), 0) == 0           # kNN <= 0: keep all (here: none)
    assert L.l3d_match_stride(fresh.h) == 1
    assert L.l3d_match_pairs(fresh.h, 1, p(pairs), p(F), C.c_float(0.25), 33) == 0           # kNN > 32: keep-all passes + per-row cut (round 2)
    assert L.l3d_match_pairs(fresh.h, 1, p(pairs), p(F), C.c_float(0.25), 5) == 0           # F = 0: valid call, no matches
    counts, total = fresh.match_counts()
    assert total == 0
    assert L.l3d_get_pair_matches(fresh.h, 3, p(counts), p(counts)) == -1
    assert L.l3d_rdd(fresh.h, 0, C.c_longlong(0), None, None, None, 10, None, None, None, None) == -1
    fresh.close()


def test_knn_above_32_vs_reference_wrapper(loaded, scene, ref):
    """kNN > 32 (beyond the fused kernel's per-row key list; the reference accepts any kNN, cudawrapper.cu:637-645): the keep-all
    passes + per-row cut must give the reference wrapper's matches, in its pop order (overlap descending)."""
    knn = 40
    pairs = np.array(PAIRS[:2], np.int32)
    loaded.set_views(util.scene_descs(scene), scene.segs)        # earlier tests put other scenes into the shared context
    loaded.match_pairs(pairs, util.pair_F(scene, pairs), 0.05, knn)       # low threshold: rows longer than 32 exist
    nlong = 0
    for p, (src, tgt) in enumerate(PAIRS[:2]):
        counts, recs = loaded.pair_matches(p, len(scene.segs[src]))
        check_lists(counts, recs, ref(f"knn40/{src}_{tgt}"), what=(src, tgt))
        assert counts.max() <= knn
        nlong += int((counts > 32).sum())
    assert nlong > 0, "the test scene must have rows with more than 32 matches"


def test_dense_batch_equals_single_launches(loaded, scene):
    """l3d_match_dense_pairs (all view pairs in one launch) writes exactly what l3d_match_dense writes pair by pair"""
    import torch
    loaded.set_views(util.scene_descs(scene), scene.segs)
    pairs = np.array(PAIRS, np.int32)
    F = util.pair_F(scene, pairs)
    deps, ovs = [], []
    for (s, t) in PAIRS:
        ns, nt = len(scene.segs[s]), len(scene.segs[t])
        deps.append(torch.full((ns * nt * 4,), 7.0, dtype=torch.float32, device="cuda"))
        ovs.append(torch.full((ns * nt,), 7.0, dtype=torch.float32, device="cuda"))
    loaded.match_dense_pairs(pairs, F, 0.25, [d.data_ptr() for d in deps], [o.data_ptr() for o in ovs])
    loaded.sync()
    for i, (s, t) in enumerate(PAIRS):
        ns, nt = len(scene.segs[s]), len(scene.segs[t])
        d1, o1 = loaded.match_dense(s, t, F[i], 0.25, ns, nt)
        assert np.array_equal(util.bits(deps[i].cpu().numpy()), util.bits(d1.reshape(-1)))
        assert np.array_equal(util.bits(ovs[i].cpu().numpy()), util.bits(o1.reshape(-1)))


@pytest.mark.parametrize("kind", ["sideways", "forward", "edge", "rolled"])
def test_level1_prefilter_never_drops(gpu_ctx, ref, kind):
    """the pencil-parameter pre-filter (k_pair_arcs, l3d_device.cuh) with the epipole at infinity, inside the image, near its border
    and with a rolled camera: same matches as the unmodified reference kernel + host kNN pass (which evaluate every cell), both
    directions; horizontal / vertical / tiny segments and segments through the epipole added on purpose"""
    sc = util.level1_scene(kind)
    gpu_ctx.set_views(util.scene_descs(sc), sc.segs)
    pairs = np.array([(0, 1), (1, 0)], np.int32)
    for epi, knn in ((0.25, 10), (0.05, 32)):
        gpu_ctx.match_pairs(pairs, util.pair_F(sc, pairs), epi, knn)
        tot = 0
        for p, (s, t) in enumerate(pairs):
            counts, recs = gpu_ctx.pair_matches(p, len(sc.segs[s]))
            # only an exact tie in the k-th place may differ (DESIGN section 2: the reference pops an unordered heap)
            check_lists(counts, recs, ref(f"level1_{kind}_{epi}_{knn}/{s}_{t}"), what=(kind, s, t, epi))
            tot += int(counts.sum())
        assert tot > 1000          # not vacuous
