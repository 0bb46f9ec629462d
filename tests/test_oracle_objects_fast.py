"""The whole-array contour model (oracle/refport.py:contour_records, remove_invalid_objects_fast) against the per-contour
closed form (contour_objects, remove_invalid_objects) it restates: per contour the same area, pixel count, mask sum and
fill (through the sum of its pixel indices), and the same output for every configuration, with and without a
segmentation mask.  That is what lets the fast model stand in for the oracle at 1080p and 4K
(tests/test_gpu_objects_fullsize.py).  The frame generators below are shared with that file."""
import os
import sys

import numpy as np
import pytest
from scipy import ndimage as ndi

from oracle import refport as R

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
from make_golden import OBJ_CFGS  # noqa: E402


# ---- frames ---------------------------------------------------------------------------------------------------------

def blobby(rng, h, w, sigma=None, q=None):
    """thresholded low-pass noise with grey values 1..255: components of every size, holes, islands in holes"""
    x = ndi.gaussian_filter(rng.random((h, w)), sigma if sigma is not None else rng.choice([1.5, 3.0, 6.0]))
    on = x > np.quantile(x, q if q is not None else rng.choice([0.4, 0.5, 0.7]))
    return (on * rng.integers(1, 256, (h, w))).astype(np.uint8)


def salt(rng, h, w, p):
    """random sites with density p, grey values 1..255 (p ~ 0.41: both classes near their percolation thresholds)"""
    return ((rng.random((h, w)) < p) * rng.integers(1, 256, (h, w))).astype(np.uint8)


def checker(h, w, phase=0):
    """one diagonal-only foreground component (8-connected) around one-pixel holes (4-connected background)"""
    yy, xx = np.indices((h, w))
    return (((yy + xx + phase) % 2 == 0) * 255).astype(np.uint8)


def rings(h, w, levels, cy=None, cx=None):
    """concentric square 1-px rings on a 2-px pitch around (cy, cx): ``levels`` nested sets, the innermost one pixel"""
    cy = h // 2 if cy is None else cy
    cx = w // 2 if cx is None else cx
    R_ = levels - 1
    yy, xx = np.indices((h, w))
    r = np.maximum(np.abs(yy - cy), np.abs(xx - cx))
    return (((r <= R_) & ((R_ - r) % 2 == 0)) * 255).astype(np.uint8)


def serpentine(h, w, pitch=2, block=0):
    """one 1-px path through every ``pitch``-th row, turning at alternate ends; ``block`` > 0 hangs a filled square of that
    side on its last row, so the component's area (and its fate) depends on the whole path being one set"""
    a = np.zeros((h, w), np.uint8)
    rows = list(range(0, max(1, h - block), pitch))
    for k, y in enumerate(rows):
        a[y, :] = 255
        if k + 1 < len(rows):
            a[y:rows[k + 1] + 1, w - 1 if k % 2 == 0 else 0] = 255
    if block:
        a[rows[-1]:rows[-1] + block, :block] = 255
    return a


def segmask_for(rng, h, w):
    """blobby 0 / 255 segmentation mask, or grey-valued noise"""
    if rng.random() < 0.7:
        return ((ndi.gaussian_filter(rng.random((h, w)), 6.0) > 0.5) * 255).astype(np.uint8)
    return rng.integers(0, 256, (h, w), dtype=np.uint8)


def handmade_objects():
    """hand-made nesting: ring with an island that has its own hole, 1-pixel-wide parts, objects on the image border,
    diagonal contacts (8-connected foreground / 4-connected background), areas either side of 100.  -> alpha, segmask"""
    h, w = 96, 128
    a = np.zeros((h, w), np.uint8)
    a[10:70, 10:90] = 200
    a[20:60, 20:80] = 0            # hole
    a[30:50, 30:60] = 150          # island in the hole
    a[35:45, 38:52] = 0            # its own hole
    a[38:42, 42:48] = 90           # island in that
    a[0:12, 100:128] = 255         # touches the border: area (11 * 27) > 100
    a[80:90, 5:15] = 77            # 10 x 10: contour area 81 < 100
    a[80:91, 30:41] = 77           # 11 x 11: contour area 100
    for k in range(15):            # diagonal chain: 8-connected, area 0
        a[75 + k, 60 + k] = 255
    a[70, 95] = 255                # diagonal contact with the big ring's corner pixel (69, 89)?  no: isolated pixel
    a[70, 90] = 255                # this one touches (69, 89) diagonally: joins the ring
    seg = np.zeros((h, w), np.uint8)
    seg[:, :70] = 255
    return a, seg


def seeded_frame(kind, seed):
    """frames up to 200 x 300 (the noisy kinds smaller: the per-contour oracle labels the frame once per contour)"""
    rng = np.random.default_rng(1000 * (KINDS.index(kind) + 1) + seed)
    if kind == "blobby":
        h, w = rng.integers(8, 201), rng.integers(8, 301)
        a = blobby(rng, h, w)
        if seed % 3 == 0:
            a[rng.random((h, w)) < 0.01] = 200
    elif kind == "salt":
        h, w = rng.integers(4, 101), rng.integers(4, 151)
        a = salt(rng, h, w, rng.uniform(0.3, 0.7))
    elif kind == "checker":
        h, w = rng.integers(2, 61), rng.integers(2, 91)
        a = checker(h, w, seed % 2)
        if seed % 3 == 1:          # bites out of it: holes merge into larger ones and open to the outside
            a[rng.random((h, w)) < 0.05] = 0
    elif kind == "rings":
        h, w = rng.integers(20, 201), rng.integers(20, 301)
        a = rings(h, w, int(rng.integers(2, 70)), rng.integers(0, h), rng.integers(0, w))
        if seed % 2:               # grow the rings into discs here and there: areas either side of 100
            a = np.maximum(a, (blobby(rng, h, w, 3.0, 0.8) > 0) * np.uint8(255))
    else:
        h, w = rng.integers(6, 201), rng.integers(6, 301)
        a = serpentine(h, w, int(rng.integers(2, 5)), int(rng.integers(0, 14)))
        if seed % 3 == 0:          # specks on it and between its rows
            a[rng.random(a.shape) < 0.05] = 255
        if seed % 2:
            a = a.T.copy()
    return a, segmask_for(rng, *a.shape)


KINDS = ["blobby", "salt", "checker", "rings", "serpentine"]


# ---- tests ----------------------------------------------------------------------------------------------------------

def per_contour(objs, seg, idx):
    """(area, pixels, mask sum, index sum) of every contour of the per-contour closed form, sorted"""
    return sorted((float(area), int(f.sum()), int(seg[f].astype(np.int64).sum()), float(idx[f].sum())) for f, area in objs)


def check_frame(a, seg):
    h, w = a.shape
    objs = R.contour_objects(a > 0)
    idx = np.arange(h * w, dtype=np.float64).reshape(h, w)      # sums of pixel indices: exact, and they identify the fill
    rec = R.contour_records(a > 0, seg, idx)[0]
    got = sorted(zip(rec["area"].tolist(), rec["count"].tolist(), rec["segsum"].tolist(), rec["score"].tolist()))
    assert got == per_contour(objs, seg, idx)
    assert np.all((rec["depth"] % 2 == 0) == rec["hole"])
    for cfg in OBJ_CFGS:
        for s in (None, seg):
            out, r = R.remove_invalid_objects_fast(cfg, a, s, return_records=True)
            assert R.decision_margin(r) > 1e-9
            assert np.array_equal(out, R.remove_invalid_objects(cfg, a, s, objs)), (cfg, s is None)
    return len(objs)


@pytest.mark.parametrize("i", range(6))
def test_fast_model_on_golden(golden, i):
    """the reference's own outputs (tests/golden/objects.npz), all configurations, with and without a segmask"""
    g = golden("objects")
    a, seg = g[f"alpha_{i}"], g[f"seg_{i}"]
    for c, cfg in enumerate(OBJ_CFGS):
        assert np.array_equal(R.remove_invalid_objects_fast(cfg, a), g[f"self_{i}_{c}"]), c
        assert np.array_equal(R.remove_invalid_objects_fast(cfg, a, seg), g[f"seg_{i}_{c}"]), c
    check_frame(a, seg)


def test_fast_model_on_handmade_shapes():
    a, seg = handmade_objects()
    check_frame(a, seg)


@pytest.mark.parametrize("kind", KINDS)
def test_fast_model_equals_per_contour_model(kind):
    """80 seeded frames of each kind; every contour and every output equal"""
    contours = [check_frame(*seeded_frame(kind, seed)) for seed in range(80)]
    assert max(contours) >= 50                  # the kinds do produce many contours


@pytest.mark.parametrize("levels", [1, 2, 64, 65, 66, 130])
def test_fast_model_nesting_depth(levels):
    """concentric rings: as many nested contours as levels, every one of them in the records"""
    n = 2 * levels + 3
    a = rings(n, n, levels)
    rec = R.contour_records(a > 0, a, np.ones(a.shape))[0]
    assert len(rec["area"]) == levels and rec["depth"].max() == levels
    check_frame(a, np.full_like(a, 255))


def test_fast_model_degenerate_frames():
    for a in (np.zeros((7, 9), np.uint8), np.full((7, 9), 255, np.uint8), np.full((1, 1), 3, np.uint8),
              np.zeros((1, 5), np.uint8), checker(1, 9), checker(9, 1)):
        check_frame(a, np.full_like(a, 200))
