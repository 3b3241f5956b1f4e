"""Records what the parity tests compare against when they run the UNMODIFIED reference (oracle/_ref, built from the reference
sources by oracle/Makefile), so that the tests need nothing outside the repository:

    python tests/golden/make_ref_outputs.py cpu tests/golden/ref_outputs_cpu_v1.npz    # clustering.cc and the verbatim CPU pipeline
    python tests/golden/make_ref_outputs.py gpu ref_outputs_gpu_v1.npz                 # the reference kernels: needs a B200

Bit-exact comparisons are stored as SHA-256 digests of the canonical bytes, toleranced ones as a fixed, seeded sample of the
values (tests/util.py: stage_record, pick).  Every entry is keyed by the test that reads it.
"""
import os
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from line3dpp_b200 import synth          # noqa: E402
from oracle import pyoracle as po        # noqa: E402
from tests import nvm_util as nu         # noqa: E402
from tests import util                   # noqa: E402

MATCH_PAIRS = [(0, 1), (0, 4), (2, 3), (5, 1), (7, 6)]          # tests/test_match_gpu.py PAIRS


def txt_record(path):
    """a result text file as numbers: count + seeded sample"""
    v = np.array(open(path).read().split(), float)
    return {"txt_n": np.int64(len(v)), "txt_smp": v[util.pick(len(v))]}


# ---------------------------------------------------------------------------------------------- CPU: clustering.cc, line3D.cc (CPU path)
def cpu_records():
    ref = po.ref_lib("nofma")
    assert ref is not None and po.ref_full_lib("cpu") is not None, "needs oracle/_ref"
    out = {}
    rng = np.random.default_rng(1)                                    # test_cpu.py::test_oracle_cluster_vs_reference_clustering_cc_live
    for n, m in [(10, 30), (500, 4000), (2000, 3000)]:
        ei, ej = rng.integers(0, n, m).astype(np.int32), rng.integers(0, n, m).astype(np.int32)
        ew = rng.choice(np.linspace(0.5, 1.0, 23), m).astype(np.float32)
        out[f"cluster_live/{n}_{m}"] = {"labels": po.cluster(ref.ref_cluster, ei, ej, ew, n, )}
    # test_ref_full_cpu.py::test_oracle_host_logic_vs_verbatim_line3d_cc
    for V, N, nb, collin, knn in [(8, 300, "ring2", -1.0, 10), (10, 250, "ring3", 2.0, 10), (6, 200, "ring2", -1.0, 0)]:
        sc = synth.make_scene(V, N, 7, nb, collinear=collin > 0)
        with tempfile.TemporaryDirectory() as d:
            R = po.RefFullPipeline(False, False, "cpu", folder=d)
            R.add_scene(sc)
            R.match_images(knn=knn)
            R.reconstruct(3, False, collin)
            rec = util.dump_record(R, sc.cam_ids, [len(s) for s in sc.segs], collin=collin > 0, exact_scores=False)
            rec.update(txt_record(os.path.join(d, R.save(d, txt=True) + ".txt")))
        out[f"host_logic/{V}_{N}_{nb}_{collin}_{knn}"] = rec
    return out


# ---------------------------------------------------------------------------------------------- GPU: the reference kernels on a B200
def gpu_records():
    ref = po.ref_lib("nofma")
    assert ref is not None and ref.ref_device_count() > 0, "needs oracle/_ref and a GPU"
    out = {}
    # tests/test_match_gpu.py
    scene = synth.make_scene(8, 700, 11, "dense")
    for s, t in MATCH_PAIRS:
        pi = util.pair_inputs(scene, s, t)
        dep, ov, _ = po.match_dense(ref.ref_match_dense, pi["ls"], pi["lt"], pi["F"], pi["Rs"], pi["Rt"], pi["Cs"], pi["Ct"], 0.25)
        sel = np.flatnonzero(ov.reshape(-1) > 0.25)
        smp = sel[util.pick(len(sel))]
        out[f"dense/{s}_{t}"] = {"ov_sha": util.sha(util.bits(ov)), "dep_sha": util.sha(util.bits(dep)), "nsel": np.int64(len(sel)),
                                 "cells": smp, "dep": dep.reshape(-1, 4)[smp]}

    def lists(tag, pairs, epi, knn, sc=scene):
        for s, t in pairs:
            pi = util.pair_inputs(sc, s, t)
            c, o, tot, _ = po.match_lines(ref.ref_match_lines, pi["ls"], pi["lt"], pi["F"], pi["Rs"], pi["Rt"], pi["Cs"], pi["Ct"], s, t, epi, knn)
            assert tot == c.sum()
            out[f"{tag}/{s}_{t}"] = {"counts": c.astype(np.uint8), "list_sha": util.list_sha(c, o), "tie_sha": util.tie_sha(c, o)}
            if tag == "topk":
                out[f"{tag}/{s}_{t}"]["row_sha"] = util.row_shas(c, o)
    lists("topk", MATCH_PAIRS, 0.25, 10)
    lists("keep_all", MATCH_PAIRS[:3], 0.25, 0)
    lists("knn40", MATCH_PAIRS[:2], 0.05, 40)
    for kind in ("sideways", "forward", "edge", "rolled"):
        sc = util.level1_scene(kind)
        for epi, knn in ((0.25, 10), (0.05, 32)):
            lists(f"level1_{kind}_{epi}_{knn}", [(0, 1), (1, 0)], epi, knn, sc)
    sc = synth.make_scene(6, 250, 13, "ring2")
    P = po.OraclePipeline(False, True, backend=ref)
    P.add_scene(sc)
    P.match_images(knn=-1)
    rec = util.dump_record(P, sc.cam_ids, None, recon=False)
    assert P.reconstruct(3, False) == 0
    rec["num_lines"] = np.int64(P.num_lines())
    out["keep_all_pipeline"] = rec
    # tests/test_collinear_gpu.py
    cs = util.collinear_scene()
    for t in (0.5, 2.0, 6.0):
        rec = {}
        for v, segs in enumerate(cs.segs):
            if len(segs):
                Cm, _ = po.collinear(ref.ref_collinear, segs, t)
                rec[f"v{v}_sha"], rec[f"v{v}_sum"] = util.sha(Cm), np.int64(Cm.sum())
        out[f"collinear/{t}"] = rec
    sc = synth.make_scene(12, 500, 93, "ring3", collinear=True)
    for diffusion, collin_t in [(False, 2.0), (True, 2.0), (True, 5.0)]:
        P = po.OraclePipeline(False, True, backend=ref)
        P.add_scene(sc)
        P.match_images()
        assert P.reconstruct(3, diffusion, collin_t) == 0
        out[f"collin_links/{diffusion}_{collin_t}"] = util.dump_record(P, sc.cam_ids, [len(s) for s in sc.segs], matching=False, collin=True)
    # tests/test_pipeline_gpu.py
    sc = synth.make_scene(14, 500, 31, "ring3")
    for diffusion in (False, True):
        P = po.OraclePipeline(False, True, backend=ref)
        P.add_scene(sc)
        assert P.match_images() == 0
        if not diffusion:
            out["pipeline/match"] = util.dump_record(P, sc.cam_ids, None, recon=False)
        assert P.reconstruct(3, diffusion) == 0
        out[f"pipeline/recon_{diffusion}"] = util.dump_record(P, sc.cam_ids, None, matching=False)
    ei, ej, ew, n = util.rdd_graph()
    ri, rj, rw, _ = po.rdd(ref.ref_rdd, ei, ej, ew, n)
    out["rdd"] = {"idx_sha": util.sha(ri.astype(np.int64), rj.astype(np.int64)), "w_sha": util.sha(util.bits(rw))}
    inp = nu.load_inputs()
    P = po.OraclePipeline(True, 1, backend=ref)
    nu.add_all(P.add_view, inp)
    assert P.match_images() == 0 and P.reconstruct(3, False) == 0
    out["pipeline/nvm"] = util.dump_record(P, range(inp["V"]), None)
    # tests/test_optimize_gpu.py
    sc = synth.make_scene(12, 500, 96, "ring3", noise_px=1.0)
    for diffusion in (False, True):
        P = po.OraclePipeline(False, True, backend=ref)
        P.add_scene(sc)
        P.match_images()
        assert P.reconstruct(3, diffusion, -1.0, True, 250) == 0
        rec = util.dump_record(P, sc.cam_ids, None, matching=False)
        rec["opt_summary"] = P.opt_summary()
        out[f"ceres/{diffusion}"] = rec
    P = po.OraclePipeline(True, 1, backend=ref)
    nu.add_all(P.add_view, inp)
    assert P.match_images() == 0 and P.reconstruct(3, False, -1.0, True, 250) == 0
    rec = util.dump_record(P, range(inp["V"]), None, matching=False)
    rec["opt_summary"] = P.opt_summary()
    out["ceres/nvm"] = rec
    # tests/test_ref_full_gpu.py: the reference's whole pipeline, CUDA path
    assert po.ref_full_lib("gpu") is not None
    for diffusion, collin, knn in [(False, -1.0, 10), (True, -1.0, 10), (True, 2.0, 10), (False, -1.0, 0)]:
        sc = synth.make_scene(12, 600, 41, "ring3", collinear=collin > 0)
        with tempfile.TemporaryDirectory() as d:
            R = po.RefFullPipeline(False, True, "gpu", folder=d)
            R.add_scene(sc)
            R.match_images(knn=knn)
            R.reconstruct(3, diffusion, collin)
            out[f"full/{diffusion}_{collin}_{knn}"] = util.dump_record(R, sc.cam_ids, [len(s) for s in sc.segs], collin=collin > 0)
    with tempfile.TemporaryDirectory() as d:
        R = po.RefFullPipeline(True, True, "gpu", folder=d)
        nu.add_all(R.add_view, inp)
        R.match_images()
        R.reconstruct(3, False)
        rec = util.dump_record(R, range(inp["V"]), [len(s) for s in inp["segs"]])
        name = R.save(d, txt=True)
        rec.update(txt_record(os.path.join(d, name + ".txt")))
        rec["txt_name"] = name
        out["full/nvm"] = rec
        R.reconstruct(3, True)
        out["full/nvm_diffusion"] = util.dump_record(R, range(inp["V"]), [len(s) for s in inp["segs"]])
    return out


if __name__ == "__main__":
    recs = cpu_records() if sys.argv[1] == "cpu" else gpu_records()
    util.save_records(sys.argv[2], recs)
    print(sys.argv[2], os.path.getsize(sys.argv[2]), "bytes,", len(recs), "records")
