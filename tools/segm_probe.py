"""Wall clock of core.test.segm_results (device paste + RLE, the D2H of the runs and building the RLE dicts) against the
reference's host loop (lib/core/test.py:793-847 without pycocotools' encode: cv2.resize + threshold + paste + the
Fortran-order copy) on tests/segm_cases.py segm_case("a"): 100 detections, 800 x 1199, M = 28, 81 class-specific masks
already on the device.  Also the kernel time of the RLE (count + scan + emit) and of the dense paste, from CUDA events.

    python tools/segm_probe.py [--iters N] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from detectron.pytorch_b200 import ops
from detectron.pytorch_b200.core import test as T
from oracle import segm as oseg
from tests.segm_cases import segm_case


def host_loop(c, cv2):
    M = c["M"]
    boxes = oseg.expand_boxes_int(c["ref_boxes"], M)
    padded = np.zeros((M + 2, M + 2), np.float32)
    out, i = [], 0
    for j in range(1, c["num_classes"]):
        for _ in range(len(c["cls_boxes"][j])):
            padded[1:-1, 1:-1] = c["masks"][i, j]
            x1, y1, x2, y2 = boxes[i]
            w, h = max(x2 - x1 + 1, 1), max(y2 - y1 + 1, 1)
            mask = np.array(cv2.resize(padded, (int(w), int(h))) > 0.5, dtype=np.uint8)
            im = np.zeros((c["im_h"], c["im_w"]), np.uint8)
            x_0, x_1 = max(x1, 0), min(x2 + 1, c["im_w"]); y_0, y_1 = max(y1, 0), min(y2 + 1, c["im_h"])
            im[y_0:y_1, x_0:x_1] = mask[y_0 - y1:y_1 - y1, x_0 - x1:x_1 - x1]
            out.append(np.array(im[:, :, np.newaxis], order="F"))
            i += 1
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    c = segm_case("a")
    kw = dict(num_classes=c["num_classes"], resolution=c["M"], cls_specific_mask=True, thresh_binarize=0.5)
    masks, boxes = torch.from_numpy(c["masks"]).cuda(), torch.from_numpy(c["ref_boxes"]).cuda()
    ch = oseg.channels_for([len(b) for b in c["cls_boxes"][1:]], True)
    H, W = c["im_h"], c["im_w"]
    for _ in range(5):
        T.segm_results(c["cls_boxes"], masks, boxes, H, W, **kw)
        ops.segm_paste(masks, ch, boxes, H, W)
    torch.cuda.synchronize()
    t = []
    for _ in range(a.iters):
        t0 = time.perf_counter()
        T.segm_results(c["cls_boxes"], masks, boxes, H, W, **kw)          # ends with a blocking D2H of the runs
        t.append(time.perf_counter() - t0)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    ch_t = torch.from_numpy(ch.astype(np.int32)).cuda()
    ev[0].record()
    for _ in range(a.iters):
        ops.segm_paste(masks, ch_t, boxes, H, W)
    ev[1].record()
    torch.cuda.synchronize()
    t_rle = []
    for _ in range(a.iters):
        t0 = time.perf_counter()
        ops.segm_rle(masks, ch_t, boxes, H, W)
        t_rle.append(time.perf_counter() - t0)
    res = {"case": "segm_case('a')", "detections": int(len(ch)), "image": [H, W], "M": c["M"],
           "segm_results_ms_median": 1e3 * float(np.median(t)), "segm_results_ms_min": 1e3 * float(np.min(t)),
           "segm_rle_call_ms_median": 1e3 * float(np.median(t_rle)),
           "segm_paste_kernel_ms": ev[0].elapsed_time(ev[1]) / a.iters,
           "gpu": torch.cuda.get_device_name(0)}
    try:
        res["power_limit"] = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader"], stdout=subprocess.PIPE,
                                            text=True, timeout=30).stdout.strip()
    except Exception as exc:  # noqa: BLE001
        res["power_limit"] = "unknown (%s)" % exc
    try:
        import cv2
        cv2.ipp.setUseIPP(False)
        th = []
        for _ in range(3):
            t0 = time.perf_counter()
            host_loop(c, cv2)
            th.append(time.perf_counter() - t0)
        res["host_loop_ms_median"] = 1e3 * float(np.median(th))
    except ImportError:
        res["host_loop_ms_median"] = None
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        ops.segm_rle(masks, ch_t, boxes, H, W)
        ops.segm_paste(masks, ch_t, boxes, H, W)
        torch.cuda.synchronize()
    res["kernels_us"] = {e.key: round(e.device_time_total, 1) for e in prof.key_averages() if "segm" in e.key}
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
