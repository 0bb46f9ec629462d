"""oracle/refport.py:laplace_residual, the oracle-free check of regionfill's Laplace solve, and toprow_fill, the closed-form
solution of that solve when every pixel but the top row is masked.  Both stand in for scipy's spsolve at sizes where the
direct solve is too slow (tests/test_gpu_bgmodel_fullsize.py)."""
import numpy as np
from scipy.fft import dct, idct

from oracle import refport as R
from video_unscreen_b200 import synth


def toprow_fill(g, h):
    """regionfill (factor 1.0) of an h x len(g) plane whose mask is every pixel but row 0, with g as row 0.  D is separable:
    nn counts in-image neighbours, so D = L_x (+) L_y with path-graph Laplacians.  The DCT-II basis diagonalises L_x
    (eigenvalue mu_k = 2 - 2 cos(pi k / w)), and per mode the rows solve (2 + mu) a_y = a_(y-1) + a_(y+1) with a_0 = g_k
    and a_h = a_(h-1) (the bottom border): a_y = g_k cosh(t (h - 1/2 - y)) / cosh(t (h - 1/2)), 2 cosh t = 2 + mu."""
    g = np.asarray(g, np.float64)
    w = g.size
    gk = dct(g, type=2, norm="ortho")
    t = np.arccosh(1.0 + (1.0 - np.cos(np.pi * np.arange(w) / w)))
    y = np.arange(h, dtype=np.float64)[:, None]
    a, b = t * (h - 0.5 - y), t * (h - 0.5)              # a, b >= 0: cosh(a) / cosh(b) without overflow
    ratio = np.exp(a - b) * (1.0 + np.exp(-2.0 * a)) / (1.0 + np.exp(-2.0 * b))
    return idct(gk * ratio, type=2, norm="ortho", axis=1)


def test_laplace_residual_of_direct_solves():
    """small on spsolve's fills (a person-like hole, holes on every border and corner, salt, all but the top row, all but one
    pixel), for one plane and for planes stacked; a 1e-6 change to one filled pixel shows"""
    h, w = 90, 160
    rng = np.random.default_rng(5)
    img = synth.textured_background(h, w, seed=3)
    plane = img[:, :, 1].astype(np.float64) + rng.random((h, w))
    masks = [synth.ellipse_mask(h, w, 80, 50, 30, 35)]
    m = np.zeros((h, w), bool)
    m[:12, :20] = m[:12, 140:] = m[80:, :15] = m[85:, 150:] = m[40:50, :9] = m[30:60, 155:] = True
    masks += [m, rng.random((h, w)) < 0.3]
    m = np.ones((h, w), bool)
    m[0] = False
    masks.append(m)
    m = np.ones((h, w), bool)
    m[37, 101] = False
    masks.append(m)
    for m in masks:
        x = R.regionfill(plane, m)
        res = R.laplace_residual(x, plane, m)
        assert res <= 1e-9, res
        x3 = np.stack([x, R.regionfill(img[:, :, 0], m), R.regionfill(img[:, :, 2], m)])
        assert R.laplace_residual(x3, np.stack([plane, img[:, :, 0], img[:, :, 2]]), m) <= 1e-9
        ys, xs = np.nonzero(m)
        for j in (0, len(ys) // 2, len(ys) - 1):
            bad = x.copy()
            bad[ys[j], xs[j]] += 1e-6
            assert R.laplace_residual(bad, plane, m) >= 1e-6
    # outside the mask only the boundary data counts; an empty mask has nothing to check
    x = R.regionfill(plane, masks[0])
    assert R.laplace_residual(np.where(masks[0], x, 0.0), plane, masks[0]) == R.laplace_residual(x, plane, masks[0])
    assert R.laplace_residual(plane, plane, np.zeros((h, w), bool)) == 0.0


def test_toprow_fill_is_the_direct_solve():
    for h, w in ((60, 97), (41, 128), (2, 33)):
        g = np.random.default_rng(h).random(w) * 255
        plane = np.zeros((h, w))
        plane[0] = g
        m = np.ones((h, w), bool)
        m[0] = False
        want = R.regionfill(plane, m)
        got = toprow_fill(g, h)
        assert np.abs(got - want).max() <= 1e-9
        assert R.laplace_residual(got, plane, m) <= 1e-9
