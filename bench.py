#!/usr/bin/env python
"""bench.py — headline benchmark of the Line3D++ matching hot path on B200 (contract: see DESIGN.md "Measurement").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--scaling weak|strong] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Metric: matched line-pairs/sec = (source segment, target segment) pair evaluations per second of the epipolar matching
+ fused kNN selection (unit of work of SURVEY.md §8(d)); every unordered view pair is evaluated once.
Workload (BASELINE.json configs[3]): synthetic 1000 views x 3000 segments/view per GPU, ring +-5 visual neighbours
(5000 view pairs, 4.5e10 pair evaluations per GPU).  Weak scaling: N GPUs match a ring of N*1000 views; every rank
owns 1000 views, one NCCL all-gather of the per-view segment lists makes all views resident, then each rank matches
the view pairs whose source view it owns (no other collective on the data path).

`--scaling strong` keeps the ring at 1000 views for every N (BASELINE.json configs[3] "sharded 1/2/4/8"): every rank owns
1000/N views and matches the pairs whose source view it owns.

One step = all-gather (N>1) + per-segment pre-pass + one fused match/top-k launch over this rank's pairs.
  value : device-timed, inputs already in HBM.
  e2e   : same step through the C ABI with HOST buffers: H2D of this rank's segments from pinned memory, match,
          D2H of the per-row counts and kNN record slots into pinned memory (l3d_match_pairs_host: chunked, the copy
          of a finished chunk overlaps the arithmetic of the next).
`--dump-outputs DIR` writes what the last timed step computed (see dump_outputs) as DIR/<name>.npy; the inputs are seeded, so two
builds of the project can be compared output for output.
`--impl reference` times the reference's CPU/OpenMP matching path (oracle port of matchingCPU, line3D.cc:900-1015;
line3D.cc itself cannot be compiled in this image) on the host cores, on a bounded sample of the same workload.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

VIEWS_PER_GPU, SEGS_PER_VIEW, RING, KNN, EPI = 1000, 3000, 5, 10, 0.25      # VIEWS_PER_GPU becomes 1000 / N with --scaling strong
SCALING = "weak"
FLOP_PER_PAIR_EVAL = 100.0     # algorithmic FP32 flop per pair evaluation (SURVEY.md §8(d), DESIGN.md "Roofline")
DENSE_BYTES_PER_CELL = 20.0    # float4 depths + float overlap per cell (cudawrapper.cu:226-251)
RDD_BYTES_PER_NNZ = 20.0       # P val + col idx + W val + transpose slot + P' store (SURVEY.md §8(d))


def dist_env():
    return int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))


# ---------------------------------------------------------------------------------------------- clocks sampler
class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md 'clocks' line)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm = [float(r[1]) for r in self.rows if len(r) > 8 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) > 8 and r[2].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows if len(r) > 8 for n, v in zip(names, r[5:9]) if v.lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


# ---------------------------------------------------------------------------------------------- workload
def build_rank_workload(rank: int, world: int):
    """This rank's views (global ids rank*1000 ..), the camera blocks of ALL views and this rank's view-pair list."""
    from line3dpp_b200 import synth
    V = VIEWS_PER_GPU * world
    # one global scene definition; each rank only materialises the segments of its own views
    t0 = time.time()
    scene = synth.make_scene(V, SEGS_PER_VIEW, 1004, f"ring{RING}") if world == 1 else None
    if scene is None:
        scene = synth.make_scene_views(V, SEGS_PER_VIEW, 1004, f"ring{RING}", range(rank * VIEWS_PER_GPU, (rank + 1) * VIEWS_PER_GPU))
    pairs = synth.view_pairs(scene.neighbors)
    from line3dpp_b200 import shard
    mine = shard.rank_pairs(pairs, rank, world, V)        # pairs whose SOURCE view this rank owns
    F = np.zeros((len(mine), 9), np.float32)
    for i, (s, t) in enumerate(mine):
        F[i] = synth.fundamental(scene.K[s], scene.R[s], scene.t[s], scene.K[t], scene.R[t], scene.t[t]).astype(np.float32).reshape(9)
    return scene, mine, F, time.time() - t0


def make_descs(scene, nsegs):
    from line3dpp_b200 import capi, synth
    RtKinv, C = synth.camera_blocks(scene)
    V = scene.num_views
    return capi.make_view_descs(scene.cam_ids, [scene.width] * V, [scene.height] * V, nsegs, RtKinv, C, C,
                                np.zeros(V, np.float32), np.zeros(V, np.float32))


# ---------------------------------------------------------------------------------------------- reference arm / cpu baseline
def cpu_matching_sample(seconds_target: float = 12.0, threads: int | None = None):
    """Times the oracle port of the reference CPU/OpenMP matching path (matchingCPU, double) on view pairs of the bench
    workload until ~seconds_target of wall time is used.  Returns (pair_evals_per_s, cores, sample description)."""
    from line3dpp_b200 import synth
    from oracle import pyoracle as po
    po.build(ref=False)
    sc = synth.make_scene(12, SEGS_PER_VIEW, 1004, f"ring{RING}")
    RtKinv, C = synth.camera_blocks(sc)
    pairs = synth.view_pairs(sc.neighbors)
    fn = po.lib().orc_match_lines_f64
    # Thread count: all the host threads the box reports (nproc) AND half of them (one per physical core when SMT is on) are both
    # timed on the same sample, each for half of the budget; the FASTER one is the baseline (the reference gets its best case),
    # both rates are reported.  No calibration shots, no per-box tuning.
    nproc = len(os.sched_getaffinity(0)) or (os.cpu_count() or 1)
    cands = [threads] if threads else sorted({nproc, max(1, nproc // 2)}, reverse=True)
    s, t = pairs[0]                       # one untimed pair: thread pool start-up, page faults
    F0 = synth.fundamental(sc.K[s], sc.R[s], sc.t[s], sc.K[t], sc.R[t], sc.t[t])
    results = []
    for cores in cands:
        po.set_threads(cores)
        po.match_lines(fn, sc.segs[s], sc.segs[t], F0, RtKinv[s], RtKinv[t], C[s], C[t], int(s), int(t), EPI, KNN, f64=True)
        done, t_used, n, rates = 0, 0.0, 0, []
        budget = seconds_target / len(cands)
        wall0 = time.perf_counter()
        while t_used < budget and time.perf_counter() - wall0 < 3.0 * budget:
            for (s_, t_) in pairs:
                F = synth.fundamental(sc.K[s_], sc.R[s_], sc.t[s_], sc.K[t_], sc.R[t_], sc.t[t_])
                ms = po.match_lines(fn, sc.segs[s_], sc.segs[t_], F, RtKinv[s_], RtKinv[t_], C[s_], C[t_], int(s_), int(t_), EPI, KNN, f64=True)[3]
                t_used += ms * 1e-3      # the port's own steady_clock around matching (LSD / I/O / Python glue excluded, BASELINE.md §2)
                done += len(sc.segs[s_]) * len(sc.segs[t_]); n += 1
                rates.append(len(sc.segs[s_]) * len(sc.segs[t_]) / (ms * 1e-3))
                if t_used >= budget:
                    break
        results.append((done / t_used, cores, n, done, t_used, float(np.std(rates) / np.mean(rates)) if rates else 0.0))
    best = max(results)
    detail = "; ".join(f"{c} threads: {v:.3g} pair-evals/s over {n} view pairs ({d:.3g} evaluations, {tu:.1f} s, per-pair rsd {100 * r:.0f} %)" for v, c, n, d, tu, r in results)
    return best[0], best[1], (f"view pairs of {SEGS_PER_VIEW}x{SEGS_PER_VIEW} segments of the bench workload, matchingCPU double path, OpenMP over source segments; "
                              f"{detail}; reported: the faster thread count")


def ref_cuda_sample(scene, npairs: int = 6):
    """B-CUDA of BASELINE.md: the reference's OWN CUDA matching path on this B200 — the unmodified match_lines_GPU
    (kernel + dense D2H of 20 B per pair evaluation + host priority-queue pass, cudawrapper.cu:549-658) from the stock
    nvcc build oracle/_ref/libl3dref_default.so, staged like matchingGPU (line3D.cc:1040-1074), on view pairs of the
    bench workload.  Part of the baseline leg (checker code, never on the product path); None if oracle/_ref is absent."""
    try:
        from line3dpp_b200 import synth
        from oracle import pyoracle as po
        ref = po.ref_lib("default")
        if ref is None or ref.ref_device_count() <= 0:
            return None
        RtKinv, C = synth.camera_blocks(scene)
        f32 = lambda a: np.ascontiguousarray(a, np.float32)
        done, ms_total = 0, 0.0
        for i in range(npairs + 1):
            s, t = 0 + i, 1 + i
            F = synth.fundamental(scene.K[s], scene.R[s], scene.t[s], scene.K[t], scene.R[t], scene.t[t])
            _, _, _, ms = po.match_lines(ref.ref_match_lines, scene.segs[s], scene.segs[t], f32(F), f32(RtKinv[s]), f32(RtKinv[t]), f32(C[s]), f32(C[t]),
                                         int(s), int(t), EPI, KNN)
            if i == 0:
                continue                      # warm-up (CUDA context, first cudaMallocPitch)
            ms_total += ms
            done += len(scene.segs[s]) * len(scene.segs[t])
        return {"value": done / (ms_total * 1e-3), "unit": "pair-evals/s", "kind": "reference (unmodified cudawrapper.cu, stock nvcc flags, sm_100a)",
                "sample": f"{npairs} view pairs of {SEGS_PER_VIEW}x{SEGS_PER_VIEW} segments, per-pair wall time of match_lines_GPU incl. its uploads/downloads and host kNN pass"}
    except Exception as e:   # noqa
        return {"error": str(e)[:200]}


def run_reference(args):
    rank, _, world = dist_env()
    if rank != 0:
        return 0
    per_step = []
    sample = ""
    cores = os.cpu_count() or 1
    for i in range(args.warmup + args.steps):
        budget = max(2.0, min(30.0, 150.0 / max(args.steps + args.warmup, 1)))
        v, cores, sample = cpu_matching_sample(budget)
        if i >= args.warmup:
            per_step.append(v)
    value = float(np.mean(per_step))
    pe_step = 4.5e10 * (max(world, 1) if SCALING == "weak" else 1)
    line = {"impl": "reference", "metric": "matched_line_pairs_per_sec", "value": value, "unit": "pair-evals/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": pe_step / value * 1e3,
            "higher_is_better": True, "scaling": SCALING, "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "value_rsd_over_steps": float(np.std(per_step) / value) if len(per_step) > 1 else None,
            "config": workload_config(args.gpus),
            "cpu_baseline": {"value": value, "unit": "pair-evals/s", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": "pair-evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "note": "reference CPU/OpenMP matching path (oracle port of line3D.cc:900-1015; line3D.cc needs Eigen/OpenCV/Boost, absent here); "
                    "ms_per_step is the time the full step's pair evaluations would take at this rate"}
    print(json.dumps(line))
    return 0


def workload_config(n):
    V = n * VIEWS_PER_GPU
    how = f"{VIEWS_PER_GPU} views x {SEGS_PER_VIEW} segments per GPU" if SCALING == "weak" else f"1000 views x {SEGS_PER_VIEW} segments in total, {VIEWS_PER_GPU} views per GPU"
    return {"workload": f"BASELINE.json configs[3]: synthetic {how}, ring +-{RING} neighbours, "
                        f"kNN={KNN}, epi_overlap={EPI}; {n} GPU(s) -> ring of {V} views, {V * RING} view pairs",
            "views": V, "segments_per_view": SEGS_PER_VIEW, "view_pairs": V * RING, "knn": KNN,
            "epi_overlap": EPI, "sharding": f"views sharded over {n} GPU(s), one NCCL all-gather of segment lists" if n > 1 else "single GPU",
            "l2": "flushed between timed steps (256 MiB write); outputs (3.6 GB/step) exceed L2"}


# ---------------------------------------------------------------------------------------------- our arm
def run_ours(args):
    import torch
    import torch.distributed as dist
    from line3dpp_b200 import capi

    rank, local_rank, world = dist_env()
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            print(json.dumps({"error": f"--gpus {args.gpus} needs torchrun with {args.gpus} ranks"}))
            return 2
    torch.cuda.set_device(local_rank)
    # rank 0 prints ONE JSON line: the "NCCL version ..." banner goes to stdout unless NCCL's log is pointed elsewhere (measured on the
    # 2-GPU box: banner with NCCL_DEBUG unset, none with NCCL_DEBUG=WARN + NCCL_DEBUG_FILE=/dev/stderr)
    os.environ.setdefault("NCCL_DEBUG", "WARN")
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    ctx = capi.Context(local_rank)
    st = torch.cuda.ExternalStream(ctx.stream)

    scene, pairs, F, gen_s = build_rank_workload(rank, world)
    V = scene.num_views
    lo, hi = rank * VIEWS_PER_GPU, (rank + 1) * VIEWS_PER_GPU
    nsegs = [SEGS_PER_VIEW] * V
    my = np.concatenate([scene.segs[v] for v in range(lo, hi)]).astype(np.float32)
    assert my.shape == (VIEWS_PER_GPU * SEGS_PER_VIEW, 4), my.shape   # equal-sized shards: all_gather_into_tensor
    descs = make_descs(scene, nsegs)
    host_my = torch.from_numpy(my).pin_memory()
    with torch.cuda.stream(st):
        dev_my = host_my.to("cuda", non_blocking=True)
        dev_all = torch.empty((V * SEGS_PER_VIEW, 4), dtype=torch.float32, device="cuda") if world > 1 else dev_my
        flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    ctx.sync()

    def step_device():
        """inputs resident in HBM -> matches resident in HBM"""
        with torch.cuda.stream(st):
            if world > 1:
                dist.all_gather_into_tensor(dev_all, dev_my)
            ctx.set_views_flat(descs, dev_all.data_ptr(), True)
            ctx.match_pairs(pairs, F, EPI, KNN)

    rows_total = int(len(pairs)) * SEGS_PER_VIEW
    E2E_CHUNKS = int(os.environ.get("L3D_E2E_CHUNKS", "32"))
    state = {"counts": None, "recs": None, "total": 0}

    def step_e2e():
        """host buffers in -> host buffers out, through the C ABI"""
        with torch.cuda.stream(st):
            if world > 1:
                dev_my.copy_(host_my, non_blocking=True)
                dist.all_gather_into_tensor(dev_all, dev_my)
                ctx.set_views_flat(descs, dev_all.data_ptr(), True)
            else:
                ctx.set_views_flat(descs, host_my.data_ptr(), False)
            if state["counts"] is None:         # page-locked output arrays of the whole job (the host-side match store)
                state["counts"] = torch.empty(rows_total, dtype=torch.int32).pin_memory()
                state["recs"] = torch.empty(rows_total * KNN * 24, dtype=torch.uint8).pin_memory()
            # match + download in one C-ABI call: the D2H of every finished chunk overlaps the arithmetic of the next one
            ctx.match_pairs_host(pairs, F, state["counts"].data_ptr(), state["recs"].data_ptr(), EPI, KNN, E2E_CHUNKS)

    def barrier():
        ctx.sync()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        barrier()
        ms = []
        for _ in range(steps):
            with torch.cuda.stream(st):
                flush.fill_(1)                     # evict L2 between timed steps (not timed)
            ctx.sync()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0 = time.perf_counter()
            e0.record(st)
            fn()
            e1.record(st)
            ctx.sync()
            wall = (time.perf_counter() - t0) * 1e3
            ms.append((e0.elapsed_time(e1), wall))
        barrier()
        return ms

    sampler = ClockSampler(local_rank)
    launches0 = ctx.launch_count()
    if rank == 0:
        sampler.start()
    dev_ms = timed(step_device, args.steps, args.warmup)
    clocks = sampler.stop() if rank == 0 else None
    launches = (ctx.launch_count() - launches0) / (args.steps + args.warmup)
    pe_local = ctx.match_pair_evals()
    if args.dump_outputs:
        dump_outputs(ctx, scene, pairs, args.dump_outputs, f"rank{rank}_" if world > 1 else "")
    e2e_ms = timed(step_e2e, args.steps, max(args.warmup, 1) + 1)   # +1: first call allocates the pinned output buffers
    assert ctx.match_total_rows() == rows_total
    state["total"] = int(state["counts"].sum().item())              # emitted matches, counted from what arrived on the host

    # ---- roofline legs measured live (rank 0): FP32 peak probe + HBM-bound dense kernel
    extra = {}
    LEAN = bool(os.environ.get("L3D_BENCH_LEAN"))       # scaling sweeps: only the step itself (no roofline legs / baselines, which belong to the N=1 line)
    if rank == 0 and not LEAN:
        extra = roofline_legs(ctx, st, scene, torch)
        try:    # REF_CPU semantics on the GPU (matchingCPU's double arithmetic, k_match_topk_f64): the f64-vs-f64 figure next to the CPU arm
            npf = min(len(pairs), 500)
            Fd = F[:npf].astype(np.float64)
            with torch.cuda.stream(st):
                ctx.match_pairs_f64(pairs[:npf], Fd, EPI, KNN)
            ctx.sync()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(st)
            with torch.cuda.stream(st):
                ctx.match_pairs_f64(pairs[:npf], Fd, EPI, KNN)
            e1.record(st); ctx.sync()
            extra.setdefault("extras", {})["match_f64"] = {"kernel": "k_match_topk_f64 (REF_CPU semantics: matchingCPU's double arithmetic)", "view_pairs": npf,
                                                           "pair_evals_per_sec": npf * SEGS_PER_VIEW * SEGS_PER_VIEW / (e0.elapsed_time(e1) * 1e-3), "ms": e0.elapsed_time(e1)}
        except Exception as e:   # noqa
            extra.setdefault("extras", {})["match_f64"] = {"error": str(e)[:200]}

    dev_total = sum(m[0] for m in dev_ms)
    e2e_total = sum(max(m) for m in e2e_ms)          # e2e includes host-side waits: take max(device, wall) per step
    t = torch.tensor([dev_total, e2e_total, float(pe_local), float(state["total"])], dtype=torch.float64, device="cuda")
    if world > 1:
        tmax = t.clone(); dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        tsum = t.clone(); dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
        dev_total, e2e_total, pe_all, matches_all = tmax[0].item(), tmax[1].item(), tsum[2].item(), tsum[3].item()
    else:
        pe_all, matches_all = float(pe_local), float(state["total"])
    if rank == 0:
        ms_step = dev_total / args.steps
        value = pe_all / (ms_step * 1e-3)
        e2e_step = e2e_total / args.steps
        h2d = int(my.nbytes + len(pairs) * (8 + 36) + V * 232)
        d2h = int(rows_total * 4 + rows_total * KNN * 24)          # per-row counts + fixed-slot records, all of it copied
        fp32_peak = extra.get("fp32_peak_tflops")
        achieved_tf = pe_all / world * FLOP_PER_PAIR_EVAL / (ms_step * 1e-3) / 1e12
        peaks = load_peaks()
        line = {
            "metric": "matched_line_pairs_per_sec", "value": value, "unit": "pair-evals/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": SCALING, "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": workload_config(args.gpus),
            "emitted_matches_per_sec": matches_all / (ms_step * 1e-3),
            "e2e": {"value": pe_all / (e2e_step * 1e-3), "unit": "pair-evals/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": e2e_step},
            "gpu_launches": launches,
            "clocks": clocks,
            "roofline": {"kernel": "k_match_topk", "bound": "fp32", "achieved": achieved_tf, "peak": fp32_peak, "unit": "TFLOP/s",
                         "frac": (achieved_tf / fp32_peak) if fp32_peak else None,
                         "peak_source": "FFMA probe kernel run live in this process (MEASURED_PEAKS.json has no FP32 non-tensor figure)",
                         "peak_nominal": nominal_fp32_tflops(clocks),
                         "frac_of_nominal": (achieved_tf / nominal_fp32_tflops(clocks)) if nominal_fp32_tflops(clocks) else None,
                         "algorithmic_flop_per_pair_eval": FLOP_PER_PAIR_EVAL,
                         "hbm_frac": (pe_all / world * 0.1 / (ms_step * 1e-3) / 1e9) / peaks["hbm_gbs"],
                         "accounting": "achieved = pair evaluations x 100 flop (SURVEY 8d: what a kernel that evaluates every cell spends) / step time; "
                                       "since round 2 k_match_topk only visits the cells inside a row's arc windows (~11 % of them), so the figure is "
                                       "throughput in brute-force-equivalent flops, not executed flops - `executed` is what the SMs issued",
                         "executed": committed_capture("k_match_topk"),
                         "traffic": committed_traffic("k_match_topk"),
                         "traffic_note": "DRAM read+write bytes per launch from the committed ncu --set full capture of this command (profiles/traffic.json); "
                                         "algorithmic output is 24 B per emitted match + 4 B per (pair,row) count"},
            "roofline_hbm": extra.get("roofline_hbm"),
            "extras": extra.get("extras"),
            "peaks": peaks,
        }
        if not LEAN:
            cpu_v, cores, sample = cpu_matching_sample(20.0)
            line["cpu_baseline"] = {"value": cpu_v, "unit": "pair-evals/s", "cores": cores, "kind": "port", "sample": sample}
            line["ref_cuda_baseline"] = ref_cuda_sample(scene)
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    # tensors allocated under the context's stream must die before the stream does
    del dev_my, dev_all, flush, host_my
    state.clear()
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    ctx.close()
    sys.stdout.flush()
    return 0


def dump_outputs(ctx, scene, pairs, out_dir, prefix="", nsample=32):
    """The match result the timed step leaves for its caller (l3d_match_pairs: per source segment of every view pair its match
    count and kNN records), as float arrays: the number of matches of every view pair, and for a fixed, seeded sample of nsample
    view pairs the full lists - counts, target segment ids, overlaps and the four depths, with -1 in every field of an empty slot
    (a match has a positive overlap and positive depths).  About 27 MB for 32 pairs of 3000 x 3000 segments."""
    os.makedirs(out_dir, exist_ok=True)
    counts, _ = ctx.match_counts()
    off = ctx.pair_row_offsets(len(pairs))
    csum = np.concatenate([[0], np.cumsum(counts, dtype=np.int64)])
    out = {"matches_per_pair": (csum[off[1:]] - csum[off[:-1]]).astype(np.float64)}
    sel = np.sort(np.random.default_rng(0).choice(len(pairs), min(nsample, len(pairs)), replace=False))
    lists = [ctx.pair_matches(int(p), len(scene.segs[pairs[p][0]])) for p in sel]
    empty = [np.arange(r.shape[1])[None, :] >= c[:, None] for c, r in lists]
    out["sample_pairs"] = pairs[sel].astype(np.float64)
    out["sample_counts"] = np.stack([c for c, _ in lists]).astype(np.float32)
    out["sample_tgt_seg"] = np.stack([np.where(e, -1.0, r["tgt_seg"]) for e, (_, r) in zip(empty, lists)])
    out["sample_overlap"] = np.stack([np.where(e, -1.0, r["overlap"]).astype(np.float32) for e, (_, r) in zip(empty, lists)])
    out["sample_depths"] = np.stack([np.where(e[..., None], -1.0, np.stack([r[f] for f in ("d_p1", "d_p2", "d_q1", "d_q2")], -1)).astype(np.float32)
                                     for e, (_, r) in zip(empty, lists)])
    for name, a in out.items():
        np.save(os.path.join(out_dir, f"{prefix}{name}.npy"), a)


def nominal_fp32_tflops(clocks):
    """148 SMs x 128 FP32 lanes x 2 flop x the SM clock sampled under load (74.5 TFLOP/s at 1965 MHz), next to the live probe"""
    try:
        import torch
        sms = torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count
        mhz = float((clocks or {}).get("sm_mhz") or (clocks or {}).get("sm_max_mhz") or 0.0)
        return sms * 128 * 2 * mhz * 1e6 / 1e12 if mhz > 0 else None
    except Exception:   # noqa
        return None


def committed_capture(kernel: str):
    """warp instructions / issue utilisation per launch of `kernel` from the committed ncu capture (profiles/traffic.json), or None"""
    try:
        d = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))[kernel]
        return {k: d[k] for k in ("warp_instructions", "issue_active_pct", "capture") if k in d}
    except Exception:   # noqa
        return None


def committed_traffic(kernel: str):
    """DRAM bytes per launch of `kernel` from the committed ncu capture (profiles/traffic.json), or None"""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))[kernel]["bytes_per_launch"]
    except Exception:   # noqa
        return None


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "source": "MEASURED_PEAKS.json (of measured)"}
    return {"hbm_gbs": 6650.0, "source": "B200_PROFILING.md fallback (of fallback)"}


def roofline_legs(ctx, st, scene, torch):
    """HBM-bound leg: the dense-contract kernel (20 B written per pair evaluation), timed with CUDA events on the
    launching stream over outputs larger than L2; plus the FP32 FFMA peak probe."""
    out = {}
    try:
        out["fp32_peak_tflops"] = ctx.fp32_peak_tflops()
    except Exception as e:   # noqa
        out["fp32_peak_tflops"] = None
    Ns = Nt = SEGS_PER_VIEW
    nbuf = 64                                           # 64 view pairs = 64 x 180 MB of output in ONE launch (l3d_match_dense_pairs): never L2 resident
    dep = [torch.empty(Ns * Nt * 4, dtype=torch.float32, device="cuda") for _ in range(nbuf)]
    ov = [torch.empty(Ns * Nt, dtype=torch.float32, device="cuda") for _ in range(nbuf)]
    from line3dpp_b200 import synth
    dpairs = np.array([(0, 1 + i) for i in range(nbuf)], np.int32)
    F = np.stack([synth.fundamental(scene.K[0], scene.R[0], scene.t[0], scene.K[t], scene.R[t], scene.t[t]).astype(np.float32).reshape(9) for t in range(1, 1 + nbuf)])
    for rep in range(2):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(st)
        ctx.match_dense_pairs(dpairs, F, EPI, [d.data_ptr() for d in dep], [o.data_ptr() for o in ov])
        e1.record(st)
        ctx.sync()
        ms_batch = e0.elapsed_time(e1) / nbuf
    for rep in range(2):                                # the reference's own granularity: one launch per view pair
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(st)
        for i in range(8):
            ctx.match_dense(0, 1 + i, F[i], EPI, Ns, Nt, dev_ptrs=(dep[i].data_ptr(), ov[i].data_ptr()))
        e1.record(st)
        ctx.sync()
        ms_single = e0.elapsed_time(e1) / 8
    ms = ms_batch
    peaks = load_peaks()
    gbs = Ns * Nt * DENSE_BYTES_PER_CELL / (ms * 1e-3) / 1e9
    out["roofline_hbm"] = [{"kernel": "k_match_dense_batch (64 view pairs per launch)", "bound": "hbm", "achieved": gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                            "frac": gbs / peaks["hbm_gbs"], "traffic": None, "ms_per_pair": ms, "ms_per_pair_one_launch_per_pair": ms_single,
                            "frac_one_launch_per_pair": Ns * Nt * DENSE_BYTES_PER_CELL / (ms_single * 1e-3) / 1e9 / peaks["hbm_gbs"],
                            "algorithmic_bytes_per_pair_eval": DENSE_BYTES_PER_CELL, "cells_per_pair": Ns * Nt,
                            "pair_evals_per_sec": Ns * Nt / (ms * 1e-3)}]
    del dep, ov
    # diffusion (SpMV-like, HBM-bound): banded random symmetric affinity graph, 2M rows, ~32M entries, 10 iterations
    try:
        rng = np.random.default_rng(7)
        n, deg = 2_000_000, 8
        a = np.repeat(np.arange(n, dtype=np.int64), deg)
        # banded like the real affinity matrix: local ids follow (view, segment) order and matches join nearby views
        b = np.clip(a + rng.integers(-3000, 3001, n * deg), 0, n - 1)
        keep = a != b
        key = np.unique(np.minimum(a[keep], b[keep]) * n + np.maximum(a[keep], b[keep]))
        a, b = (key // n).astype(np.int32), (key % n).astype(np.int32)
        w = rng.uniform(0.5, 1.0, len(a)).astype(np.float32)
        ei, ej, ew = np.concatenate([a, b]), np.concatenate([b, a]), np.concatenate([w, w])
        iters = 10
        _, _, _, ms = ctx.rdd(n, ei, ej, ew, iters)
        _, _, _, ms = ctx.rdd(n, ei, ej, ew, iters)
        nnz = len(ei)
        gbs = iters * (RDD_BYTES_PER_NNZ * nnz + 8.0 * n) / (ms * 1e-3) / 1e9
        out["roofline_hbm"].append({"kernel": "k_rdd_step+k_rdd_normalize", "bound": "hbm", "achieved": gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                                    "frac": gbs / peaks["hbm_gbs"], "traffic": None, "ms_per_iteration": ms / iters, "rows": n, "nnz": nnz,
                                    "algorithmic_bytes_per_nnz_per_iteration": RDD_BYTES_PER_NNZ})
    except Exception as e:   # noqa
        out["roofline_hbm"].append({"kernel": "k_rdd_step", "error": str(e)[:200]})
    # the two optional stages around the path (SURVEY.md §8f-3 / §8f-4), timed once each; not part of `value`
    out["extras"] = {}
    try:
        cells = float(scene.num_views) * SEGS_PER_VIEW * SEGS_PER_VIEW      # every view of the context (remote shards included)
        ctx.find_collinear(2.0, 0); ctx.find_collinear(0.0, 0)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(st); entries = ctx.find_collinear(2.001, 0); e1.record(st); ctx.sync()
        ms = e0.elapsed_time(e1)
        ctx.find_collinear(0.0, 0)
        out["extras"]["collinear"] = {"kernel": "k_collinear (count + scan + fill, all views in one launch pair)", "views": scene.num_views, "cells": cells, "ms": ms,
                                      "cells_per_sec": cells / (ms * 1e-3), "list_entries": entries, "threshold_px": 2.0}
    except Exception as e:   # noqa
        out["extras"]["collinear"] = {"error": str(e)[:200]}
    try:
        from tests import nvm_util as nu
        before, after, ptr, res = nu.load_opt_pairs()
        cams, shift = nu.optimizer_inputs(nu.load_inputs())
        rep = 40
        p = np.tile(before + np.tile(shift, 2), (rep, 1))
        pp = np.concatenate([[0], np.cumsum(np.tile(np.diff(ptr), rep))])
        cam = np.tile(res[:, 0].astype(np.int32), rep); xy = np.tile(res[:, 2:6], (rep, 1))
        for _ in range(2):
            t0 = time.time(); _, _, summ = ctx.optimize_lines(p, pp, cam, xy, cams, 250); wall = time.time() - t0
        out["extras"]["bundling"] = {"kernel": "l3d_optimize_lines (Ceres-equivalent LM, all lines per launch)", "lines": len(p), "residuals": len(cam),
                                     "ms_wall_incl_copies": wall * 1e3, "lm_iterations": int(summ[0]), "kernels": int(summ[7]),
                                     "cost_before": summ[1], "cost_after": summ[2],
                                     "input": "the reference's own result clusters (testdata/Line3D++_ref), replicated x40"}
    except Exception as e:   # noqa
        out["extras"]["bundling"] = {"error": str(e)[:200]}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--dump-outputs", metavar="DIR", default=None, help="write what the last timed step computed to DIR/<name>.npy")
    args = ap.parse_args()
    global VIEWS_PER_GPU, SCALING
    SCALING = args.scaling
    if SCALING == "strong":
        if 1000 % max(args.gpus, 1):
            print(json.dumps({"error": "--scaling strong needs a GPU count that divides 1000"}))
            return 2
        VIEWS_PER_GPU = 1000 // max(args.gpus, 1)
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
