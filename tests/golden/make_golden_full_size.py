"""Golden samples of the REFERENCE's own CUDA kernels (oracle/_ref/*.so, built by `make -C oracle ref`) at
BASELINE.json's full sizes, for the GPU tests whose outputs are too large to store whole.  Needs a GPU:

    python tests/golden/make_golden_full_size.py OUT_DIR      # then copy OUT_DIR/*.npz into tests/golden/

Inputs are regenerated from the seeds the tests use.  Each output is stored as its values (`<key>`) at the flat
indices tests/cases.py sample_index(size, seed) picks, with that seed (`<key>_seed`).  For the backward-spread test the
whole-array statistics it needs (the reference's run-to-run spread and its error against the fp64 oracle)
are computed here on the full arrays and stored as scalars.
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from detectron.pytorch_b200 import synthetic as S     # noqa: E402
from oracle import cpu as O                          # noqa: E402
from oracle import gpu_ref as G                      # noqa: E402
from tests import cases                              # noqa: E402


def sample(a, seed):
    return np.int64(seed), a.reshape(-1)[cases.sample_index(a.size, seed)]


def main(out_dir):
    os.makedirs(out_dir, exist_ok=True)
    assert torch.cuda.is_available() and G.available()
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()    # noqa: E731
    # BASELINE configs 1 and 2: forward and backward of the reference kernel on the inputs of
    # test_roi_align_baseline_cfg1_and_cfg2_full_size
    for name, cfg in (("cfg1", S.CFG1), ("cfg2", S.CFG2)):
        P, s, sr = cfg["pooled"], cfg["scale"], cfg["sampling_ratio"]
        f = S.make_features(cfg["shape"]); r = S.make_rois(cfg["rois"], cfg["shape"], s)
        dy = np.random.RandomState(1).standard_normal((cfg["rois"], cfg["shape"][1], P, P)).astype(np.float32)
        out = G.roi_align_forward(dev(f), dev(r), P, P, s, sr).cpu().numpy()
        dx = G.roi_align_backward(dev(dy), dev(r), cfg["shape"], P, P, s, sr).cpu().numpy()
        oi, ov = sample(out, 1)
        di, dv = sample(dx, 2)
        np.savez_compressed(os.path.join(out_dir, "roi_align_ref_%s.npz" % name), out_seed=oi, out=ov, dx_seed=di, dx=dv)
        print(name, "fwd == oracle on %.6f of the elements" % np.mean(out == O.roi_align_forward(f, r, P, P, s, sr)))
    # the cases of test_backward_tolerance_is_derived_from_the_reference_kernels_own_spread
    spread = {}
    for name, (shape, s, P, sr, r, seed) in cases.spread_cases().items():
        dy = np.random.RandomState(seed).standard_normal((r.shape[0], shape[1], P, P)).astype(np.float32)
        ref64 = O.roi_align_backward(dy, r, shape, P, P, s, sr, acc64=True)
        runs = [G.roi_align_backward(dev(dy), dev(r), shape, P, P, s, sr).cpu().numpy() for _ in range(4)]
        di, dv = sample(runs[0], 3)
        spread[name + "/run_to_run_max_abs"] = np.float64(max(float(np.max(np.abs(runs[i] - runs[0]))) for i in range(1, 4)))
        spread[name + "/vs_fp64_max_abs"] = np.float64(max(float(np.max(np.abs(x - ref64))) for x in runs))
        spread[name + "/dx_seed"] = di
        spread[name + "/dx"] = dv
        print(name, {k: float(v) for k, v in spread.items() if k.startswith(name) and v.ndim == 0})
    np.savez_compressed(os.path.join(out_dir, "roi_align_ref_spread.npz"), **spread)
    # the existing small-case golden files still describe these kernels: forward bit-exact, dX within 1e-5
    for name in sorted(cases.ROI_CASES):
        c, f, r, dy = cases.roi_case(name)
        P, s, sr = c["P"], c["scale"], c["sr"]
        g = np.load(os.path.join(ROOT, "tests", "golden", "roi_align_xfrom_%s.npz" % name))
        out = G.roi_align_forward(dev(f), dev(r), P, P, s, sr).cpu().numpy()
        dx = G.roi_align_backward(dev(dy), dev(r), c["shape"], P, P, s, sr).cpu().numpy()
        print(name, "golden out bit-exact:", np.array_equal(out, g["out"]), "golden dx max abs diff: %.3g" % np.max(np.abs(dx - g["dx"])))
    torch.cuda.synchronize()
    print("golden written to", out_dir, sorted(os.listdir(out_dir)))


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "tests", "golden"))
