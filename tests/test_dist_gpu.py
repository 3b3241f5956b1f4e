"""Sharded matchImages (L3DPP::Line3D::setShard, SURVEY.md §8(e)): the multi-GPU result must equal the single-GPU one
bit for bit.  Two legs: (1) both shards emulated on ONE device (always runs with `-m gpu`), (2) two real processes over
NCCL when the box has >= 2 GPUs."""
import ctypes as C
import os
import socket
import subprocess
import sys
import textwrap

import numpy as np
import pytest

from line3dpp_b200 import line3d, synth

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _dump(L, scene):
    out = {"est": L.estimates(), "aff": L.affinity(raw=True), "seg3d": L.segments3d(), "resid": L.residuals()}
    out["kept"] = [L.view_matches(c, True) for c in scene.cam_ids]
    return out


def _same(a, b):
    assert a["est"][0].tobytes() == b["est"][0].tobytes() and a["est"][1].tobytes() == b["est"][1].tobytes()
    for x, y in zip(a["kept"], b["kept"]):
        assert x.tobytes() == y.tobytes()
    for x, y in zip(a["aff"], b["aff"]):
        assert x.tobytes() == y.tobytes()
    assert a["seg3d"].tobytes() == b["seg3d"].tobytes() and a["resid"].tobytes() == b["resid"].tobytes()


def test_setshard_two_shards_on_one_device_equal_unsharded():
    import torch
    from line3dpp_b200 import dist as l3dist
    scene = synth.make_scene(10, 300, 7, "ring3")
    full = line3d.Line3D(neighbors_by_worldpoints=False)
    full.add_scene(scene); full.match_images(); full.reconstruct_3d_lines(3, True)
    want = _dump(full, scene)

    seen = {}

    def make_cb(rank):
        def cb(_u, counts_dev, recs_dev, row_bounds, world, knn):
            rb = [row_bounds[i] for i in range(world + 1)]
            counts = l3dist.device_bytes(counts_dev, 4 * rb[-1], 0)
            recs = l3dist.device_bytes(recs_dev, l3dist.REC_BYTES * knn * rb[-1], 0)
            seen[rank] = (counts, recs, rb, knn)
            torch.cuda.synchronize()
            if rank == 0:                       # rank 1 ran first: pull its rows (the broadcast a real job would do)
                c1, r1, rb1, _ = seen[1]
                assert rb1 == rb
                a, b = rb[1], rb[2]
                counts[4 * a:4 * b] = c1[4 * a:4 * b]
                recs[l3dist.REC_BYTES * knn * a:l3dist.REC_BYTES * knn * b] = r1[l3dist.REC_BYTES * knn * a:l3dist.REC_BYTES * knn * b]
                torch.cuda.synchronize()
            return 0
        return l3dist._EXCHANGE_T(cb)

    shards, cbs = [], []
    for rank in (1, 0):
        L = line3d.Line3D(neighbors_by_worldpoints=False)
        L.add_scene(scene)
        cbs.append(make_cb(rank))
        L._chk(L.L.l3dpp_set_shard(L.h, rank, 2, cbs[-1], None), "setShard")
        L.match_images()
        shards.append(L)
    rb = seen[0][2]
    assert 0 < rb[1] < rb[2], "both shards must own rows"
    ev = [s.stats()["pair_evaluations"] for s in shards]
    assert sum(ev) == full.stats()["pair_evaluations"] and min(ev) > 0.3 * sum(ev)      # disjoint, complete, balanced
    L0 = shards[1]
    L0.reconstruct_3d_lines(3, True)
    _same(_dump(L0, scene), want)
    # rank 1 never received rank 0's rows: its scoring saw fewer matches, so the test would notice a no-op exchange
    assert sum(len(L0.view_matches(c, False)) for c in scene.cam_ids) > sum(len(shards[0].view_matches(c, False)) for c in scene.cam_ids)
    for L in shards + [full]:
        L.close()


def test_setshard_rejects_bad_arguments():
    from line3dpp_b200 import capi
    L = line3d.Line3D(neighbors_by_worldpoints=False)
    for rank, world in ((2, 2), (-1, 2), (0, 0)):
        with pytest.raises(capi.L3DError):
            L._chk(L.L.l3dpp_set_shard(L.h, rank, world, None, None), "setShard")
    with pytest.raises(capi.L3DError):
        L._chk(L.L.l3dpp_set_shard(L.h, 0, 2, None, None), "setShard")        # world > 1 needs an exchange function
    L._chk(L.L.l3dpp_set_shard(L.h, 0, 1, None, None), "setShard")
    L.close()


WORKER = textwrap.dedent("""
    import os, sys, numpy as np, torch, torch.distributed as dist
    sys.path.insert(0, %r)
    from line3dpp_b200 import line3d, synth, dist as l3dist
    dev = int(os.environ["LOCAL_RANK"]); torch.cuda.set_device(dev)
    dist.init_process_group("nccl", device_id=torch.device("cuda", dev))
    scene = synth.make_scene(12, 400, 9, "ring3")
    def dump(L):
        b, p = L.estimates(); s, r = L.segments3d(), L.residuals()
        return b.tobytes() + p.tobytes() + s.tobytes() + r.tobytes() + b"".join(L.view_matches(c, True).tobytes() for c in scene.cam_ids)
    full = line3d.Line3D(neighbors_by_worldpoints=False, device=dev)
    full.add_scene(scene); full.match_images(); full.reconstruct_3d_lines(3, True)
    L = line3d.Line3D(neighbors_by_worldpoints=False, device=dev)
    L.add_scene(scene)
    keep = l3dist.attach(L, dev)
    L.match_images(); L.reconstruct_3d_lines(3, True)
    assert L.stats()["pair_evaluations"] < full.stats()["pair_evaluations"], "this rank evaluated every pair"
    assert L.stats()["lines3D"] == full.stats()["lines3D"] > 50
    assert dump(L) == dump(full), "sharded result differs from the single-GPU result"
    ev = torch.tensor([L.stats()["pair_evaluations"]], device="cuda"); dist.all_reduce(ev)
    assert ev.item() == full.stats()["pair_evaluations"]
    dist.barrier(); L.close(); full.close(); dist.destroy_process_group()
    print("rank", dev, "sharded == unsharded")
""")


def test_two_process_nccl_sharded_equals_single_gpu(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    script = tmp_path / "worker.py"
    script.write_text(WORKER % ROOT)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", str(port), str(script)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, env=dict(os.environ, NCCL_DEBUG="WARN"))
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
