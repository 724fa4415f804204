"""CPU restatement of the quad-strip forward's work decomposition (detectron/pytorch_b200/csrc/roi_align_strip.cu: enum_row, the
strip geometry and the residency rules), checked for its invariants on seeded and adversarial RoIs.  No GPU, no library call:
this pins the ALGORITHM the prepass and the main kernel agree on.

Invariants:
  1. every sample (RoI, ph, pw, iy, ix) belongs to exactly one fragment (its bit in the fragment's sample mask);
  2. a fragment's taps lie inside its strip's slot (columns [s WX, s WX + SX - 1]) and inside its row window [key, end), and the
     window fits the ring (end - key <= K) -- so a fragment can always become resident;
  3. a fragment that holds all sr^2 samples of its bins is written with plain stores (red = 0); the others accumulate (red = 1),
     and exactly one of the fragments sharing a bin holds its first sample (the one whose bins the prepass zero-fills);
  4. fragments are at most 8 bins long, consecutive bins of one bin row.
"""
import numpy as np
import pytest

from detectron.pytorch_b200 import synthetic as S

f32 = np.float32
FRAG_BINS = 8


def axis_low(v, size):
    """xfrom_axis (common.cuh): low cell and validity of one sample coordinate."""
    valid = not (v < -1.0 or v > size)
    if v <= 0:
        v = f32(0)
    low = int(v)
    if low >= size - 1:
        low = size - 1
    return low, valid


def roi_axes(roi, scale, PH, PW, sr, H, W):
    """-> (yl, xl): PH * sr low rows (bin height from PH) and PW * sr adjusted low columns (bin width from PW)."""
    sw = f32(roi[1]) * f32(scale); sh = f32(roi[2]) * f32(scale)
    rw = max(f32(f32(roi[3]) * f32(scale) - sw), f32(1)); rh = max(f32(f32(roi[4]) * f32(scale) - sh), f32(1))
    bh = f32(rh / f32(PH)); bw = f32(rw / f32(PW))
    yl, xl = [], []
    for s in range(PH * sr):
        p, i = divmod(s, sr)
        vy = f32(f32(f32(p) * bh + sh) + f32(f32(f32(i + 0.5) * bh) / f32(sr)))
        yl.append(axis_low(vy, H)[0])
    for s in range(PW * sr):
        p, i = divmod(s, sr)
        vx = f32(f32(f32(p) * bw + sw) + f32(f32(f32(i + 0.5) * bw) / f32(sr)))
        lx, _ = axis_low(vx, W)
        if lx >= W - 1:
            lx = W - 2                                    # adj_axis: the last column is read as (W - 2, W - 1)
        xl.append(lx)
    return yl, xl


def strips(W, SX, WX):
    s = 1
    while (s - 1) * WX + SX < W:
        s += 1
    return s


def enum_row(yl, xl, ph, PW, sr, SX, WX, K, n_strips):
    """-> list of (strip, key, end, pw0, npw, smask, red, owner), exactly enum_row<SR> of the kernel file."""
    out = []
    i0, i1 = ph * sr, ph * sr + sr - 1
    groups = [(yl[i0], yl[i1] + 2, (1 << sr) - 1)]
    if sr == 2 and groups[0][1] - groups[0][0] > K:
        groups = [(yl[i0], yl[i0] + 2, 1), (yl[i1], yl[i1] + 2, 2)]
    xfull = (1 << sr) - 1
    for key, end, ym in groups:
        run = None                                        # [s, xm, pw0, n]

        def flush():
            nonlocal run
            if run is None:
                return
            s, xm, pw0, n = run
            smask = 1 if sr == 1 else ((xm if ym & 1 else 0) | ((xm << 2) if ym & 2 else 0))
            red = (ym != xfull) or (xm != xfull)
            out.append((s, key, end, pw0, n, smask, int(red), bool(red and (ym & 1) and (xm & 1))))
            run = None

        def push(s, xm, pw):
            nonlocal run
            if run is not None and run[0] == s and run[1] == xm and run[3] < FRAG_BINS and pw == run[2] + run[3]:
                run[3] += 1
                return
            flush()
            run = [s, xm, pw, 1]
        for pw in range(PW):
            j0, j1 = pw * sr, pw * sr + sr - 1
            s0 = min(xl[j0] // WX, n_strips - 1)
            if sr == 1 or xl[j1] + 1 <= s0 * WX + SX - 1:
                push(s0, xfull, pw)
            else:
                push(s0, 1, pw)
                push(min(xl[j1] // WX, n_strips - 1), 2, pw)
        flush()
    return out


GEOMS = [(32, 24, 48), (64, 56, 27), (64, 56, 24), (96, 80, 17)]          # (SX, WX, K): the kernel's three slot widths, TMA / cp.async ring depths


@pytest.mark.parametrize("SX,WX,K", GEOMS)
@pytest.mark.parametrize("shape,scale,P,sr,lo,hi", [
    ((1, 256, 200, 272), 0.25, 7, 2, 32, 512),            # BASELINE cfg2
    ((2, 256, 50, 84), 1 / 16, 14, 2, 64, 900),           # mask head on P4
    ((1, 32, 400, 64), 0.25, 7, 2, 16, 1590),             # whole-height boxes: y windows beyond the ring
    ((1, 32, 50, 336), 0.25, 7, 2, 16, 1300),             # whole-width boxes: bins cut by strip borders
    ((3, 32, 40, 68), 1 / 16, 7, 1, 32, 512),             # one sample per bin
    ((1, 8, 30, 9), 1 / 32, 7, 2, 32, 300),               # narrower than a slot
])
def test_fragments_cover_every_sample_once_and_fit_their_window(SX, WX, K, shape, scale, P, sr, lo, hi):
    check_fragments(SX, WX, K, shape, scale, P, P, sr, lo, hi)


@pytest.mark.parametrize("SX,WX,K", GEOMS)
@pytest.mark.parametrize("shape,scale,PH,PW,sr,lo,hi", [
    # bin rows of PW bins, PH * sr y samples -- a swapped size would miss or duplicate samples
    ((1, 32, 400, 64), 0.25, 16, 3, 2, 16, 1590),         # tall grid at the axis limit, y windows beyond the ring
    ((1, 32, 50, 336), 0.25, 3, 16, 2, 16, 1300),         # wide grid at the axis limit, bins cut by strip borders
    ((2, 32, 60, 100), 1 / 8, 7, 14, 2, 32, 700),
    ((2, 32, 60, 100), 1 / 8, 14, 7, 2, 32, 700),
    ((1, 16, 40, 68), 1 / 16, 1, 31, 1, 32, 900),         # one bin row of 31 bins: at least four fragments
    ((1, 16, 40, 68), 1 / 16, 31, 1, 1, 32, 900),
])
def test_fragments_non_square_grids(SX, WX, K, shape, scale, PH, PW, sr, lo, hi):
    check_fragments(SX, WX, K, shape, scale, PH, PW, sr, lo, hi)


def check_fragments(SX, WX, K, shape, scale, PH, PW, sr, lo, hi):
    N, C, H, W = shape
    rois = np.concatenate([S.make_rois(120, shape, scale, seed=3, min_size=lo, max_size=hi), S.make_edge_rois(shape, scale)]).astype(np.float32)
    n_strips = strips(W, SX, WX)
    assert (n_strips - 1) * WX + SX >= W                  # the last strip reaches the last column
    for roi in rois:
        yl, xl = roi_axes(roi, scale, PH, PW, sr, H, W)
        assert len(yl) == PH * sr and len(xl) == PW * sr
        assert all(0 <= y <= H - 1 for y in yl) and all(0 <= x <= W - 2 for x in xl)
        zeroed, split = [], set()                         # the prepass zero-fill list: element ph * PW + pw of the RoI's output
        for ph in range(PH):
            frags = enum_row(yl, xl, ph, PW, sr, SX, WX, K, n_strips)
            seen = {}
            for (s, key, end, pw0, npw, smask, red, owner) in frags:
                if owner:
                    zeroed += [ph * PW + pw for pw in range(pw0, pw0 + npw)]
                if red:
                    split.update(ph * PW + pw for pw in range(pw0, pw0 + npw))
                assert 1 <= npw <= FRAG_BINS and pw0 + npw <= PW and 0 <= s < n_strips
                assert ph < 32 and pw0 < 32                   # 5-bit fields of the fragment record
                assert 0 < end - key <= K, "a fragment must be able to become resident"
                assert key >= 0 and end <= H + 1              # row H is the zero row
                full = (1 << (sr * sr)) - 1
                assert (smask == full) == (red == 0)
                for pw in range(pw0, pw0 + npw):
                    for iy in range(sr):
                        for ix in range(sr):
                            if not (smask >> (iy * sr + ix)) & 1:
                                continue
                            k = (pw, iy, ix)
                            assert k not in seen, "sample evaluated twice"
                            seen[k] = (red, owner)
                            x = xl[pw * sr + ix]; y = yl[ph * sr + iy]
                            assert s * WX <= x and x + 1 <= s * WX + SX - 1, "x taps outside the slot"
                            assert key <= y and y + 2 <= end, "y taps (rows y, y + 1) outside the window"
            assert len(seen) == PW * sr * sr, "a sample is missing"
            for pw in range(PW):                            # split bins: every part accumulates, exactly one part owns the zero-fill
                parts = {seen[(pw, iy, ix)] for iy in range(sr) for ix in range(sr)}
                reds = {p[0] for p in parts}
                assert len(reds) == 1
                if reds == {1}:
                    assert seen[(pw, 0, 0)][1] is True
                    assert sum(1 for p in parts if p[1]) == 1
        assert len(zeroed) == len(set(zeroed)) and set(zeroed) == split, "every split bin is zero-filled exactly once"
        assert all(0 <= b < PH * PW for b in zeroed)
