#!/usr/bin/env python
"""bench.py -- headline benchmark of the RoIAlign hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]

A "step" is one pass of the hot path over one batch of synthetic input at BASELINE.json configs[1]:
RoIAlign (Caffe2-exact) forward + backward, 1x256x200x272 fp32 feature map, 512 RoIs, 7x7, sr=2.
One process per GPU; every rank owns its own image (feature map + its 512 RoIs) -- images shard
naturally, there is no data-path collective (SURVEY.md 8e) -- so scaling is weak and
value = (RoIs processed by all ranks) / (max over ranks of the device time of K steps).

Keys beyond the base contract:
  roofline      dominant kernel's algorithmic bytes / measured launch time vs MEASURED_PEAKS.json
  cpu_baseline  the CPU restatement of the reference kernel (oracle/, OpenMP) on this box's cores
  e2e           same metric through the reference-shaped plugin with HOST buffers (H2D + D2H timed)
  kernels       per-kernel launch times / fractions, plus the reference's own CUDA kernels
                (oracle/_ref, recompiled for sm_100a) timed on the same inputs when present
`--dump-outputs DIR` writes what the last timed step computed (rank 0) as float32 .npy files: roi_align_out.npy, the
whole forward output (512, 256, 7, 7), and grad_features_even_channels.npy, the feature-map gradient of every second
channel (1, 128, 200, 272) -- 53.5 MB in all.  The inputs are seeded, so two builds run with the same arguments can be
compared output for output.
`--impl reference` times the reference algorithm on the host cores (the reference has no CPU
RoIAlign -- functions/roi_align.py:28-29 -- so this is the op-for-op C restatement in oracle/).
"""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "RoIs/sec RoIAlign fwd+bwd (256ch,200x272,512 RoI)"
UNIT = "RoIs/s"
WORKLOAD = "RoIAlign fwd+bwd 1x256x200x272 fp32, 512 RoIs, 7x7, sampling_ratio=2 (BASELINE.json configs[1])"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--sets", type=int, default=6, help="rotating input sets (each 163 MB) so no step re-reads L2-resident data")
    ap.add_argument("--no-graph", action="store_true", help="time direct launches instead of a CUDA graph of the K steps")
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="budget of the cpu_baseline sample")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 path")
    return args


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ------------------------------------------------------------------------------------------------
# CPU arm: the oracle port on the host cores
# ------------------------------------------------------------------------------------------------
def cpu_reference_run(steps, warmup, budget_s, bounded=True):
    """Times fwd+bwd of the cfg2 workload with the C restatement (all host threads).  Returns
    (rois_per_s, ms_per_step, info).  When `bounded`, the RoI count of a step is cut so that
    (warmup + steps) steps fit in `budget_s`."""
    import numpy as np
    from detectron.pytorch_b200 import synthetic as S
    from oracle import cpu as O          # bench.py's cpu_baseline / --impl reference leg (allowed use)
    cfg = S.CFG2
    P, s, sr = cfg["pooled"], cfg["scale"], cfg["sampling_ratio"]
    f = S.make_features(cfg["shape"])
    rois = S.make_rois(cfg["rois"], cfg["shape"], s)
    dy = np.random.RandomState(1).standard_normal((cfg["rois"], cfg["shape"][1], P, P)).astype(np.float32)
    def _probe():
        t0 = time.perf_counter()
        O.roi_align_forward(f, rois[:64], P, P, s, sr)
        O.roi_align_backward(dy[:64], rois[:64], cfg["shape"], P, P, s, sr)
        return time.perf_counter() - t0                   # 64 RoIs + one dX zero-fill

    # all the host threads it can use -- but SMT siblings often hurt this memory-bound loop: keep the faster setting
    logical = os.cpu_count() or 1
    best = None
    for nt in sorted({logical, max(1, logical // 2)}, reverse=True):
        O.set_threads(nt)
        _probe()
        dtp = min(_probe(), _probe())
        if best is None or dtp < best[0]:
            best = (dtp, nt)
    O.set_threads(best[1])
    probe = best[0]
    n_rois = cfg["rois"]
    if bounded:
        est_full = probe * cfg["rois"] / 64.0
        if est_full * (steps + warmup) > budget_s:
            n_rois = int(max(16, min(cfg["rois"], cfg["rois"] * budget_s / (est_full * (steps + warmup)))))
    r, d = rois[:n_rois], dy[:n_rois]
    for _ in range(warmup):
        O.roi_align_forward(f, r, P, P, s, sr); O.roi_align_backward(d, r, cfg["shape"], P, P, s, sr)
    t0 = time.perf_counter()
    for _ in range(steps):
        O.roi_align_forward(f, r, P, P, s, sr); O.roi_align_backward(d, r, cfg["shape"], P, P, s, sr)
    dt = time.perf_counter() - t0
    info = {"kind": "port", "cores": O.max_threads(),
            "sample": "%d steps of fwd+bwd on %d of the 512 RoIs (same 256x200x272 map), oracle/roi_ops_oracle.c with OpenMP" % (steps, n_rois)}
    return n_rois * steps / dt, dt / steps * 1e3, info


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    steps, warmup = max(1, args.steps), max(0, args.warmup)
    value, ms, info = cpu_reference_run(steps, warmup, budget_s=150.0)
    info["value"] = value
    info["unit"] = UNIT
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
            "warmup": warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": {"workload": WORKLOAD, "device": "host CPU"},
            "cpu_baseline": info,
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))
    return 0


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
def main():
    args = parse_args()
    if args.impl == "reference":
        return run_reference_arm(args)

    import numpy as np
    import torch
    import torch.distributed as dist
    from detectron.pytorch_b200 import _lib, benchutil, ops
    from detectron.pytorch_b200 import synthetic as S
    from detectron.pytorch_b200.modeling.roi_xfrom.roi_align.functions.roi_align import RoIAlignFunction

    rank, world, local = benchutil.dist_env()
    if args.gpus > 1 and world == 1:
        # convenience: relaunch under torchrun (the driver launches torchrun itself)
        os.execvp(sys.executable, [sys.executable, "-m", "torch.distributed.run", "--nnodes=1",
                                   "--nproc-per-node", str(args.gpus), "--master-addr", "127.0.0.1",
                                   "--master-port", os.environ.get("MASTER_PORT", "29533"), os.path.abspath(__file__)] + sys.argv[1:])
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the product path has no CPU fallback)")
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    if world > 1:
        import datetime
        dist.init_process_group("nccl", device_id=device, timeout=datetime.timedelta(seconds=180))
    lib = _lib.load()

    cfg = S.CFG2
    shape, P, scale, sr, R = cfg["shape"], cfg["pooled"], cfg["scale"], cfg["sampling_ratio"], cfg["rois"]
    N, C, H, W = shape
    K, Wm = args.steps, max(3, args.warmup)
    nsets = max(2, args.sets)

    # ---- synthetic inputs, resident in HBM; `nsets` independent sets are rotated so that every step
    #      reads/writes data that left L2 long ago (6 x 163 MB >> 126 MB L2)
    gen = torch.Generator(device=device); gen.manual_seed(1234 + rank)
    feats = [torch.randn(shape, generator=gen, device=device) for _ in range(nsets)]
    dys = [torch.randn((R, C, P, P), generator=gen, device=device) for _ in range(nsets)]
    rois_np = [S.make_rois(R, shape, scale, seed=100 * rank + i) for i in range(nsets)]
    rois = [torch.from_numpy(r).to(device) for r in rois_np]
    outs = [torch.empty((R, C, P, P), device=device) for _ in range(nsets)]
    dxs = [torch.empty(shape, device=device) for _ in range(nsets)]
    stream = torch.cuda.current_stream()

    ws_bytes = int(lib.b200_roi_align_workspace_bytes(N, R, H, W, P, P, sr))
    wss = [torch.empty((max(ws_bytes, 1),), dtype=torch.uint8, device=device) for _ in range(nsets)]

    def fwd(i):
        _lib.check(lib.b200_roi_align_forward_ws(feats[i].data_ptr(), scale, N, R, H, W, C, P, P, sr, rois[i].data_ptr(),
                                                 outs[i].data_ptr(), wss[i].data_ptr() if ws_bytes else None, ws_bytes,
                                                 torch.cuda.current_stream().cuda_stream), "fwd")

    bws_bytes = int(lib.b200_roi_align_backward_workspace_bytes(N, R, C, H, W, P, P, sr))
    bws = torch.empty((max(bws_bytes, 1),), dtype=torch.uint8, device=device)     # one scratch image, reused every step

    def bwd(i):
        _lib.check(lib.b200_roi_align_backward_ws(dys[i].data_ptr(), scale, N, R, H, W, C, P, P, sr, rois[i].data_ptr(),
                                                  dxs[i].data_ptr(), bws.data_ptr() if bws_bytes else None, bws_bytes,
                                                  torch.cuda.current_stream().cuda_stream), "bwd")

    def step(i):
        fwd(i % nsets); bwd(i % nsets)

    def barrier():
        if world > 1:
            dist.barrier(device_ids=[local])
        torch.cuda.synchronize()

    def timed(fn_iter, n, graph=False, collective=True):
        """device time (ms) of n calls fn_iter(i), CUDA events on the launching stream.  `collective=False`
        for measurements only some ranks take (no barrier: a rank-local barrier would deadlock the others)."""
        sync = barrier if collective else torch.cuda.synchronize
        g = None
        if graph:
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                fn_iter(0)                                   # warm lazy init outside capture
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                for i in range(n):
                    fn_iter(i)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        sync()
        e0.record()
        if g is not None:
            g.replay()
        else:
            for i in range(n):
                fn_iter(i)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        sync()
        return ms

    # ---- warm-up (untimed)
    for i in range(Wm):
        step(i)
    torch.cuda.synchronize()

    use_graph = not args.no_graph
    launches_before = _lib.launch_count()
    with benchutil.ClockSampler(gpu_index=local) as clk:
        try:
            ms_total = timed(step, K, graph=use_graph)
        except Exception as exc:  # noqa: BLE001  (graph capture unsupported -> direct launches)
            sys.stderr.write("bench: CUDA graph path failed (%s); timing direct launches\n" % exc)
            use_graph = False
            ms_total = timed(step, K, graph=False)
        # the timed steps were 0 .. K-1: keep what the last one wrote before anything else runs on these buffers
        last = (K - 1) % nsets
        dumped = (outs[last].clone(), dxs[last][:, ::2].clone()) if args.dump_outputs and rank == 0 else None
        # The timed region is only ~35 ms long (nvidia-smi samples every 100 ms): keep replaying the identical steps,
        # untimed, for another half second so that the clock / throttle samples are taken under this very load.
        t_soak = time.perf_counter()
        while time.perf_counter() - t_soak < 0.5:
            for i in range(K):
                step(i)
            torch.cuda.synchronize()
        clocks = clk.summary()
        clocks["window"] = "timed region + 0.5 s of the identical steps launched back to back (untimed)"
    launches_per_step = None
    l0 = _lib.launch_count(); step(0); launches_per_step = _lib.launch_count() - l0
    torch.cuda.synchronize()
    ms_max, units = benchutil.aggregate(ms_total, R * K, device=device)
    value = units / (ms_max * 1e-3)

    # ---- per-kernel launch times (rank-local, device-resident, rotating sets), for the roofline
    n_k = max(20, min(200, K))
    ms_fwd = timed(lambda i: fwd(i % nsets), n_k, graph=use_graph, collective=False) / n_k
    ms_bwd = timed(lambda i: bwd(i % nsets), n_k, graph=use_graph, collective=False) / n_k
    peak_gbs, peak_src = load_peaks()
    touched = benchutil.roi_align_touched_cells(rois_np[0], N, H, W, P, P, scale, sr)
    bts = benchutil.roi_align_bytes(shape, R, P, P, touched_cells=touched)
    dom = "bwd" if ms_bwd >= ms_fwd else "fwd"
    dom_ms = ms_bwd if dom == "bwd" else ms_fwd
    achieved = bts[dom] / (dom_ms * 1e-3) / 1e9
    kernels = {
        "fwd": {"ms": ms_fwd, "algorithmic_bytes": bts["fwd"], "gbs": bts["fwd"] / (ms_fwd * 1e-3) / 1e9,
                "frac_of_measured": bts["fwd"] / (ms_fwd * 1e-3) / 1e9 / peak_gbs,
                "frac_of_8TBs": bts["fwd"] / (ms_fwd * 1e-3) / 8e12, "rois_per_s": R / (ms_fwd * 1e-3)},
        "bwd": {"ms": ms_bwd, "algorithmic_bytes": bts["bwd"], "gbs": bts["bwd"] / (ms_bwd * 1e-3) / 1e9,
                "frac_of_measured": bts["bwd"] / (ms_bwd * 1e-3) / 1e9 / peak_gbs,
                "frac_of_8TBs": bts["bwd"] / (ms_bwd * 1e-3) / 8e12, "rois_per_s": R / (ms_bwd * 1e-3)},
        "touched_cells": touched, "timing": "CUDA events, %s, %d rotating input sets" % ("CUDA graph replay" if use_graph else "direct launches", nsets),
    }
    roofline = {"bound": "hbm", "kernel": "roi_align_%s" % dom, "achieved": achieved, "peak": peak_gbs, "unit": "GB/s",
                "frac": achieved / peak_gbs, "peak_source": peak_src, "traffic": None,
                "algorithmic_bytes": bts[dom], "launch_ms": dom_ms}
    traffic_file = os.path.join(ROOT, "profiles", "traffic.json")     # dram bytes per launch from the committed ncu capture
    if os.path.exists(traffic_file):
        try:
            roofline["traffic"] = json.load(open(traffic_file)).get("roi_align_%s" % dom)
        except Exception:  # noqa: BLE001
            pass

    # ---- proposal NMS (BASELINE.json configs[2]): 6000 boxes, IoU 0.7, device-resident, no host sync
    try:
        nms_boxes = [torch.from_numpy(S.make_nms_boxes(S.CFG3["boxes"], seed=i)).to(device) for i in range(4)]
        ops.nms_raw(nms_boxes[0], S.CFG3["thresh"])
        ms_nms = timed(lambda i: ops.nms_raw(nms_boxes[i % 4], S.CFG3["thresh"]), 40, collective=False) / 40
        kept = int(ops.nms_raw(nms_boxes[0], S.CFG3["thresh"])[1].item())
        kernels["nms_6000"] = {"ms": ms_nms, "boxes_per_s": S.CFG3["boxes"] / (ms_nms * 1e-3), "kept": kept,
                               "informational_bytes": benchutil.nms_bytes(S.CFG3["boxes"], kept)}
    except Exception as exc:  # noqa: BLE001
        kernels["nms_6000"] = {"error": str(exc)}

    # ---- the reference's own CUDA kernels (recompiled for sm_100a) on the same inputs, if present
    if rank == 0:
        try:
            from oracle import gpu_ref as G      # timed as a BASELINE beside ours, never on the product path
            if G.available():
                def ref_step(i):
                    j = i % nsets
                    G.roi_align_forward(feats[j], rois[j], P, P, scale, sr)
                    G.roi_align_backward(dys[j], rois[j], shape, P, P, scale, sr)
                for i in range(3):
                    ref_step(i)
                n_r = max(10, min(50, K))
                ms_ref = timed(ref_step, n_r, collective=False) / n_r
                ms_ref_f = timed(lambda i: G.roi_align_forward(feats[i % nsets], rois[i % nsets], P, P, scale, sr), n_r,
                                 collective=False) / n_r
                G.nms_gpu(nms_boxes[0], S.CFG3["thresh"])
                t0 = time.perf_counter()
                for i in range(10):
                    G.nms_gpu(nms_boxes[i % 4], S.CFG3["thresh"])       # blocking by construction (host scan)
                ms_ref_nms = (time.perf_counter() - t0) / 10 * 1e3
                kernels["reference_cuda_sm100a"] = {"fwd_bwd_ms": ms_ref, "fwd_ms": ms_ref_f, "rois_per_s": R / (ms_ref * 1e-3),
                                                    "nms_6000_ms_wall": ms_ref_nms,
                                                    "note": "reference .cu unmodified + its Python zero-fills (oracle/_ref)"}
        except Exception as exc:  # noqa: BLE001
            kernels["reference_cuda_sm100a"] = {"error": str(exc)}

    # ---- e2e: the reference-shaped plugin with HOST buffers; H2D of features/rois/dY and D2H of
    #      out/dX are inside the timed region, every step
    fn = RoIAlignFunction(P, P, scale, sr)
    with benchutil.numa_local(local):                 # pinned buffers first-touched on the GPU's NUMA node
        h_feat = torch.randn(shape).pin_memory(); h_rois = torch.from_numpy(rois_np[0]).pin_memory()
        h_dy = torch.randn((R, C, P, P)).pin_memory()
        h_out = torch.empty((R, C, P, P)).pin_memory(); h_dx = torch.empty(shape).pin_memory()
    h2d = h_feat.numel() * 4 + h_rois.numel() * 4 + h_dy.numel() * 4
    d2h = h_out.numel() * 4 + h_dx.numel() * 4

    pipe = benchutil.E2EPipeline(fn, shape, R, C, P, device, h_feat, h_rois, h_dy, h_out, h_dx)
    e2e_run = pipe.run

    e2e_run(3)
    torch.cuda.synchronize()
    K_e2e = max(5, min(K, 50))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    e2e_run(K_e2e)
    e1.record()
    torch.cuda.synchronize()
    ms_e2e = e0.elapsed_time(e1)
    barrier()
    ms_e2e_max, units_e2e = benchutil.aggregate(ms_e2e, R * K_e2e, device=device)
    try:
        pcie = benchutil.pcie_bandwidth(device, h_feat, h_dx)
        pcie["floor_ms_per_step"] = (h2d + d2h) / (pcie["duplex_gbs"] * 1e9) * 1e3
    except Exception as exc:  # noqa: BLE001
        pcie = {"error": str(exc)}
    e2e = {"value": units_e2e / (ms_e2e_max * 1e-3), "unit": UNIT, "host_link": pcie, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
           "steps": K_e2e, "ms_per_step": ms_e2e_max / K_e2e,
           "path": "RoIAlignFunction(7,7,1/4,2)(features, rois) + .backward(dY); per step: H2D of features+rois+dY from pinned "
                   "host memory, D2H of out+dX; copies of neighbouring steps overlap the kernels (3 streams, 2 slots)"}

    # ---- CPU baseline (rank 0, N == 1 only), bounded sample
    cpu_baseline = None
    if rank == 0 and world == 1:
        try:
            v, ms_cpu, info = cpu_reference_run(steps=3, warmup=1, budget_s=args.cpu_seconds)
            info.update({"value": v, "unit": UNIT, "ms_per_step": ms_cpu})
            cpu_baseline = info
        except Exception as exc:  # noqa: BLE001
            cpu_baseline = {"error": str(exc)}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": Wm,
            "ms_per_step": ms_max / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "parallelism": "dp%d (one image per GPU, no data-path collective)" % world,
                       "rois_per_gpu": R, "l2": "inputs larger than L2: %d rotating input sets x 163 MB per rank" % nsets,
                       "launch": "CUDA graph of the K steps" if use_graph else "direct launches"},
            "roofline": roofline, "cpu_baseline": cpu_baseline, "e2e": e2e,
            "gpu_launches": int(launches_per_step * K), "launches_per_step": int(launches_per_step),
            "clocks": clocks, "kernels": kernels,
        }
        print(json.dumps(line))
    if dumped is not None:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, t in zip(("roi_align_out", "grad_features_even_channels"), dumped):
            np.save(os.path.join(args.dump_outputs, name + ".npy"), t.cpu().numpy().astype(np.float32))
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
