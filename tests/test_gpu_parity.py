"""Parity of the CUDA path (through the C ABI, via the reference-shaped Python
layer) against the CPU oracle and the committed golden vectors produced by the
unmodified reference.  Bit-exact for masks / trimaps / alpha / backgrounds;
<= 1 LSB for anything that ends in cv2's HSV2BGR (tolerance: 1, SURVEY A.5)."""
import numpy as np
import pytest

from conftest import maxdiff

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

from oracle import cvmodel as M  # noqa: E402
from oracle import refport as R  # noqa: E402

BGCOL = np.array([60, 200, 40], np.uint8)
HSV2BGR_TOL = 1  # uint8 LSB


@pytest.fixture(scope="module")
def vu():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import video_unscreen_b200.unscreen.utils as U
    from video_unscreen_b200 import ops
    from video_unscreen_b200.unscreen.colorfiltering import ColorFilteringAgent
    from video_unscreen_b200.unscreen.trimap import TrimapAgent

    class NS:
        pass
    ns = NS()
    ns.U, ns.ops, ns.CF, ns.TA = U, ops, ColorFilteringAgent, TrimapAgent
    return ns


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def host(t):
    return t.cpu().numpy()


# ---- primitives ------------------------------------------------------------

def test_bgr2hsv_gray_exhaustive(vu):
    a = np.arange(1 << 24, dtype=np.uint32)
    img = np.stack([a & 255, (a >> 8) & 255, (a >> 16) & 255], -1).astype(np.uint8).reshape(4096, 4096, 3)
    assert np.array_equal(host(vu.ops.bgr2hsv(dev(img))), M.bgr2hsv(img))
    assert np.array_equal(host(vu.ops.bgr2gray(dev(img))), M.bgr2gray(img))
    hsv = img.copy()
    hsv[..., 0] %= 180
    assert np.array_equal(host(vu.ops.hsv2bgr(dev(hsv))), M.hsv2bgr(hsv))  # same truncating f32 formula


def test_pixel_kernels_ragged_sizes(vu):
    rng = np.random.default_rng(0)
    for h, w in [(1, 1), (3, 5), (7, 9), (33, 47)]:
        img = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        assert np.array_equal(host(vu.ops.bgr2hsv(dev(img))), M.bgr2hsv(img))
        assert np.array_equal(host(vu.ops.bgr2gray(dev(img))), M.bgr2gray(img))
        assert np.array_equal(host(vu.ops.inrange_color(dev(img), [10, 20, 30], [100, 200, 250])) * 255,
                              M.in_range(M.bgr2hsv(img), [10, 20, 30], [100, 200, 250]))


@pytest.mark.parametrize("k,n", [(3, 1), (3, 2), (3, 5), (4, 2), (5, 3), (7, 10), (5, 10)])
def test_morphology(vu, k, n):
    rng = np.random.default_rng(k * 31 + n)
    for shape in [(97, 131), (2, 64, 200), (5, 3)]:
        m = rng.integers(0, 256, shape, dtype=np.uint8)
        for fn, ref in ((vu.ops.dilate, M.dilate), (vu.ops.erode, M.erode)):
            got = host(fn(dev(m), k, n))
            want = ref(m, k, n) if m.ndim == 2 else np.stack([ref(x, k, n) for x in m])
            assert np.array_equal(got, want)


@pytest.mark.parametrize("shape", [(97, 131), (3, 64, 200), (5, 3), (33, 128), (40, 257)])
def test_cross_chain_and_trimap_core(vu, shape):
    rng = np.random.default_rng(sum(shape))
    m = rng.integers(0, 256, shape, dtype=np.uint8)
    m3 = m if m.ndim == 3 else m[None]
    D, E = 0, 1
    for segs in ([(D, 2), (E, 2), (E, 2), (D, 2)], [(E, 3), (D, 1)], [(D, 12)], [(E, 5)], [(D, 0), (E, 4)]):
        want = []
        for x in m3:
            for op, it in segs:
                x = M.dilate(x, 3, it) if op == D else M.erode(x, 3, it)
            want.append(x)
        got = host(vu.ops.cross_chain(dev(m), segs))
        assert np.array_equal(got.reshape(m3.shape), np.stack(want)), segs
    for r in (1, 5, 12):
        want = []
        for x in m3:
            dil, ero = M.dilate(x, 3, r), M.erode(x, 3, r)
            t = np.full(x.shape, 128, np.uint8)
            t[ero > 127] = 255
            t[dil < 128] = 0
            want.append(t)
        assert np.array_equal(host(vu.ops.trimap_core(dev(m), r)).reshape(m3.shape), np.stack(want)), r
    # fused threshold-on-load == threshold then chain
    a = rng.integers(0, 256, m3.shape, dtype=np.uint8)
    got = host(vu.ops.cf_postprocess(dev(a), dev(m3)))
    assert np.array_equal(got, np.stack([R.cf_postprocess(x, y) for x, y in zip(a, m3)]))


def test_cross_march_flat_units(vu):
    """the marching kernels' shortcut for units (112-column strips x 64-row bands) whose input is one value after the
    threshold: mattes made of constant blocks (0, below / above the threshold, 127 / 128, 255), blocks with a single
    odd pixel (in the strip's halo columns and lead-in rows too), against the oracle's morphology"""
    rng = np.random.default_rng(11)
    h, w = 200, 480
    frames = []
    for _ in range(6):
        m = np.zeros((h, w), np.uint8)
        for y0 in range(0, h, 50):
            for x0 in range(0, w, 60):
                m[y0:y0 + 50, x0:x0 + 60] = rng.choice([0, 0, 0, 60, 127, 128, 200, 255])
        for _ in range(3):
            m[rng.integers(0, h), rng.integers(0, w)] = rng.integers(0, 256)
        frames.append(m)
    frames.append(np.full((h, w), 255, np.uint8))
    frames.append(np.zeros((h, w), np.uint8))
    m3 = np.stack(frames)
    D, E = 0, 1
    for segs in ([(D, 2), (E, 2), (E, 2), (D, 2)], [(D, 5)], [(E, 5)], [(D, 2)], [(E, 1)]):
        want = []
        for x in m3:
            for op, it in segs:
                x = M.dilate(x, 3, it) if op == D else M.erode(x, 3, it)
            want.append(x)
        assert np.array_equal(host(vu.ops.cross_chain(dev(m3), segs)), np.stack(want)), segs
    for r in (1, 3, 5):
        want = []
        for x in m3:
            dil, ero = M.dilate(x, 3, r), M.erode(x, 3, r)
            t = np.full(x.shape, 128, np.uint8)
            t[ero > 127] = 255
            t[dil < 128] = 0
            want.append(t)
        assert np.array_equal(host(vu.ops.trimap_core(dev(m3), r)), np.stack(want)), r
    masks = np.where(rng.random(m3.shape) < 0.7, 255, 0).astype(np.uint8)
    got = host(vu.ops.cf_postprocess(dev(m3), dev(masks)))
    assert np.array_equal(got, np.stack([R.cf_postprocess(x, y) for x, y in zip(m3, masks)]))


@pytest.mark.parametrize("sh,sw,dh,dw", [(270, 480, 135, 240), (360, 640, 90, 160), (135, 240, 270, 480), (90, 160, 360, 640),
                                         (250, 333, 150, 200), (150, 200, 250, 333), (480, 270, 240, 135), (61, 47, 122, 94), (9, 7, 4, 3)])
def test_resize(vu, sh, sw, dh, dw):
    rng = np.random.default_rng(sh * 7 + dw)
    img = rng.integers(0, 256, (2, sh, sw, 3), dtype=np.uint8)
    msk = rng.integers(0, 256, (2, sh, sw), dtype=np.uint8)
    assert np.array_equal(host(vu.ops.resize_linear_image(dev(img), dh, dw)), np.stack([M.resize_linear(x, dw, dh) for x in img]))
    assert np.array_equal(host(vu.ops.resize_linear_mask(dev(msk), dh, dw)), np.stack([M.resize_linear(x, dw, dh) for x in msk]))
    assert np.array_equal(host(vu.ops.resize_nearest_mask(dev(msk), dh, dw)), np.stack([M.resize_nearest(x, dw, dh) for x in msk]))
    assert np.array_equal(host(vu.ops.resize_nearest_image(dev(img), dh, dw)), np.stack([M.resize_nearest(x, dw, dh) for x in img]))


def test_golden_primitives(vu, golden):
    p = golden("primitives")
    m = p["mask"]
    U = vu.U
    for k, n in [(3, 2), (3, 5), (4, 2), (5, 3), (7, 10), (5, 10)]:
        assert np.array_equal(U.dilate_mask(m, k, n), p[f"dilate_{k}_{n}"])
        assert np.array_equal(U.erode_mask(m, k, n), p[f"erode_{k}_{n}"])
    assert np.array_equal(U.get_outer_boundary(m), p["outer_boundary"])
    assert [U.exist_foreground(m, t) for t in (0.001, 0.4, 0.5, 0.6)] == list(p["exist_fg"])
    assert np.array_equal(U.is_pixel_inrange(p["img"], p["bgcolor"], (10, 100, 180)), p["inrange_color"])
    assert np.array_equal(U.is_pixel_inrange(p["img"], np.array([5, 9, 250], np.uint8), (60, 255, 255)), p["inrange_color_wide"])
    assert np.array_equal(U.is_pixel_inrange(p["img"], p["bgimg"], (20, 20, 120)), p["inrange_image"])
    assert np.array_equal(U.is_pixel_inrange(p["img"], p["bgimg"], (10, 100, 180)), p["inrange_image2"])
    for th, tw, h, w, L in p["target_sizes"]:
        assert U.get_target_size(h, w, L) == (th, tw)
    # 3-channel masks go through per-channel morphology like cv2
    m3 = np.stack([m, m[::-1].copy(), m[:, ::-1].copy()], -1)
    assert np.array_equal(U.dilate_mask(m3, 3, 2), M.dilate(m3, 3, 2))
    # long_side_input > 0 variant against the oracle
    assert np.array_equal(U.is_pixel_inrange(p["img"], p["bgcolor"], (60, 255, 255), 64), R.is_pixel_inrange(p["img"], p["bgcolor"], (60, 255, 255), 64))
    assert np.array_equal(U.is_pixel_inrange(p["img"], p["bgimg"], (20, 20, 120), 64), R.is_pixel_inrange(p["img"], p["bgimg"], (20, 20, 120), 64))


# ---- colour filtering ----------------------------------------------------------

def load_agent(vu, c, tag):
    from test_oracle_golden import cf_tables
    lb, lf, bgh = cf_tables(c, tag)
    ag = vu.CF(input_long_side=int(c[f"{tag}_L"]))
    ag.set_tables(lb, lf, bgh)
    return ag, lb, lf, bgh


@pytest.mark.parametrize("tag", ["x2", "x4", "frac", "portrait"])
def test_colorfilter_predict_golden(vu, golden, tag):
    c = golden("colorfilter")
    ag, lb, lf, bgh = load_agent(vu, c, tag)
    a, bgimg, _ = ag.forward(c[f"{tag}_frame"], c[f"{tag}_seg"], 0)
    assert np.array_equal(a, c[f"{tag}_alpha_pred"])            # bit-exact vs the reference
    assert maxdiff(bgimg, c[f"{tag}_bgimg"]) <= HSV2BGR_TOL
    a2, _, _ = ag.forward(c[f"{tag}_frame2"], c[f"{tag}_seg2"], 0)
    assert np.array_equal(a2, c[f"{tag}_alpha_pred2"])
    # pieces
    fr, seg = c[f"{tag}_frame"], c[f"{tag}_seg"]
    th, tw = R.get_target_size(*fr.shape[:2], int(c[f"{tag}_L"]))
    hl = M.resize_linear(M.bgr2hsv(fr), tw, th)
    raw, _ = ag.get_alpha_by_gmm(hl)
    assert np.array_equal(raw, c[f"{tag}_alpha_raw"])
    assert np.array_equal(ag.postprocess(raw, M.resize_linear(seg, tw, th)), c[f"{tag}_alpha_post"])
    # the tabulated (h,s,v) -> alpha volume gives the same answer
    lut3d = vu.ops.cf_build_lut3d(ag._luts_dev)
    assert np.array_equal(host(vu.ops.cf_alpha_lut3d(dev(hl), lut3d)), c[f"{tag}_alpha_raw"])


def test_colorfilter_tables_match_oracle(vu, golden):
    from video_unscreen_b200.unscreen.colorfiltering.agent import gmm_table
    c = golden("colorfilter")
    for nm in ("bg", "fg"):
        for i in range(3):
            means, covs, w = c[f"x2_{nm}{i}_means"], c[f"x2_{nm}{i}_covs"], c[f"x2_{nm}{i}_weights"]
            assert np.array_equal(gmm_table(means, np.sqrt(covs), w).numpy(), R.gmm_lut(means, covs, w))


def test_colorfilter_fit_matches_reference_fit(vu, golden):
    """iters=3 with the same numpy RNG seed reproduces the reference's fitted
    run (the EM itself is scikit-learn on both sides)."""
    c = golden("colorfilter")
    ag = vu.CF(input_long_side=int(c["x2_L"]))
    np.random.seed(0)
    a, _, _ = ag.forward(c["x2_frame"], c["x2_seg"], 3)
    assert np.array_equal(a, c["x2_alpha_fit"])
    assert ag.is_trained()


def test_colorfilter_early_outs(vu, golden):
    c = golden("colorfilter")
    fr = c["early_frame"]
    z = np.zeros(fr.shape[:2], np.uint8)
    ag = vu.CF(input_long_side=48)
    a, b, conf = ag.forward(fr, z, 0)
    assert np.array_equal(a, c["early_nofg_alpha"]) and np.array_equal(b, c["early_nofg_bg"]) and conf == 1.0
    a, b, conf = ag.forward(fr, z + 255, 0)
    assert np.array_equal(a, c["early_nobg_alpha"]) and np.array_equal(b, c["early_nobg_bg"]) and conf == 1.0


# ---- trimap ------------------------------------------------------------------------

@pytest.mark.parametrize("tag", ["x2", "x4", "frac", "portrait", "up"])
def test_trimap_golden(vu, golden, tag):
    t = golden("trimap")
    ta = vu.TA(input_long_side=int(t[f"{tag}_L"]))
    fr = t[f"{tag}_frame"]
    assert np.array_equal(ta.forward(t[f"{tag}_mask"]), t[f"{tag}_plain"])
    assert np.array_equal(ta.forward(t[f"{tag}_soft"]), t[f"{tag}_plain_soft"])
    assert np.array_equal(ta.forward(t[f"{tag}_soft"], fr, BGCOL), t[f"{tag}_withcolor"])
    assert np.array_equal(ta.forward(t[f"{tag}_soft"], fr, t[f"{tag}_bgimg"]), t[f"{tag}_withimage"])
    assert np.array_equal(ta.forward(t[f"{tag}_leak"], fr, BGCOL), t[f"{tag}_leak_withcolor"])
    assert np.array_equal(ta.forward(t[f"{tag}_ring"], fr, BGCOL), t[f"{tag}_ring_withcolor"])
    assert np.array_equal(ta.forward(t[f"{tag}_ring"], fr, t[f"{tag}_bgimg"]), t[f"{tag}_ring_withimage"])


def test_trimap_empty_and_device_tensors(vu, golden):
    t = golden("trimap")
    z = np.zeros((40, 64), np.uint8)
    out = vu.TA(input_long_side=64).forward(z, np.zeros((40, 64, 3), np.uint8), np.array([1, 2, 3], np.uint8))
    assert np.array_equal(out, t["empty_withcolor"])
    ta = vu.TA(input_long_side=int(t["x2_L"]))
    got = ta.forward(dev(t["x2_soft"]), dev(t["x2_frame"]), BGCOL)
    assert got.is_cuda and np.array_equal(host(got), t["x2_withcolor"])


# ---- compositing -------------------------------------------------------------------------

def test_composite_golden(vu, golden):
    k = golden("composite")
    U = vu.U
    fr, al, bg = k["frame"], k["alpha"], k["bg"]
    assert maxdiff(U.get_fg(fr, al, bg), k["get_fg"]) <= HSV2BGR_TOL
    assert maxdiff(U.get_bg(al, bg), k["get_bg"]) <= HSV2BGR_TOL
    assert maxdiff(U.get_fg(fr, al, bg, patch="lt128"), k["green_patch_fg"]) <= HSV2BGR_TOL
    assert maxdiff(U.get_fg(fr, al, bg, patch="eq0"), k["bg_patch_fg"]) <= HSV2BGR_TOL
    # and exactly the oracle's truncating HSV2BGR
    assert np.array_equal(U.get_fg(fr, al, bg), R.get_fg(fr, al, bg))
    assert np.array_equal(U.get_bg(al, bg), R.get_bg(al, bg))
    assert np.array_equal(U.get_fg_naive(fr, al), k["get_fg_naive"])
    assert np.array_equal(U.fuse_fgbg(fr, bg, al), k["fuse_fgbg"])
    assert np.array_equal(U.composite_fgbg(fr, al, k["newbg"]), k["composite"])
    assert np.array_equal(U.composite_fgbg(fr, al, k["newbg"], True), k["composite_ext"])
    assert np.array_equal(U.composite_fgbg(fr, al, k["tallbg"]), k["composite_tall"])
    assert np.array_equal(U.replace_blend(fr, np.stack([al] * 3, -1), bg), k["replace"])
    assert np.array_equal(U.replace_blend(fr, al, bg), k["replace"])
    assert np.array_equal(U.fuse_bg(bg, k["bg_always"], 0.1), k["fused_bg"])
    assert np.array_equal(U.bgdiff_gate(fr, k["near_bg"], al, 25), k["gate"])
    assert np.array_equal(U.binarise_dilate(al), k["binarise_dilate"])
    # patched background is returned bit-exactly when asked for
    fg, bgo = vu.ops.get_fg(dev(fr), dev(al), dev(bg), 1, want_bg=True)
    assert np.array_equal(host(bgo), R.patch_bg(bg, fr, al, "lt128"))


def test_blend_all_alpha_values(vu):
    """every (fg, alpha, bg) byte triple class: float64 sequences are bit-exact."""
    rng = np.random.default_rng(3)
    fg = rng.integers(0, 256, (256, 256, 3), dtype=np.uint8)
    bg = rng.integers(0, 256, (256, 256, 3), dtype=np.uint8)
    al = np.repeat(np.arange(256, dtype=np.uint8)[:, None], 256, 1)
    U = vu.U
    assert np.array_equal(U.replace_blend(fg, al, bg), R.replace_blend(fg, al, bg))
    assert np.array_equal(U.fuse_fgbg(fg, bg, al), R.fuse_fgbg(fg, bg, al))
    assert np.array_equal(U.get_fg_naive(fg, al), R.get_fg_naive(fg, al))
    assert np.array_equal(U.composite_fgbg(fg, al, bg), R.composite_fgbg(fg, al, bg))
    assert np.array_equal(U.get_fg(fg, al, bg), R.get_fg(fg, al, bg))


def test_replace_blend_every_triple_on_every_lane(vu):
    """The integer replace / fuse blend (blend16_int_kernel) against the float64 expression of replace.py:74-76 on ALL 2^24
    (alpha, fg, bg) byte triples, shifted so that every triple passes through each of the twelve byte positions of the
    kernel's four-pixel pattern (pairs, singles, both accumulators of the fix-up bits)."""
    n = 1 << 24
    p = np.arange(n, dtype=np.uint32)
    a, c, q = (p >> 16).astype(np.uint8), ((p >> 8) & 255).astype(np.uint8), (p & 255).astype(np.uint8)
    m = a.astype(np.float64) / 255
    want = (c.astype(np.float64) * m + q.astype(np.float64) * (1 - m)).astype(np.uint8)
    assert np.array_equal(want[:300000:4097], R.replace_blend(c[:300000:4097, None, None].repeat(3, 2), a[:300000:4097, None],
                                                              q[:300000:4097, None, None].repeat(3, 2))[:, 0, 0])
    U = vu.U
    for shift in range(4):
        ar, cr, qr, wr = (np.roll(x, shift) for x in (a, c, q, want))
        fg = dev(np.repeat(cr[:, None], 3, 1).reshape(4096, 4096, 3))
        bg = dev(np.repeat(qr[:, None], 3, 1).reshape(4096, 4096, 3))
        al = dev(ar.reshape(4096, 4096))
        got = host(U.replace_blend(fg, al, bg)).reshape(n, 3)
        for ch in range(3):
            bad = np.flatnonzero(got[:, ch] != wr)
            assert bad.size == 0, (shift, ch, bad[:5], got[bad[:5], ch], wr[bad[:5]])
        if shift == 0:
            assert np.array_equal(host(U.fuse_fgbg(fg, bg, al)).reshape(n, 3), got)


@pytest.mark.parametrize("shape,thr", [((70, 128), 25), ((64, 120), 25), ((131, 244), 10), ((9, 12), 25), ((200, 500), 254), ((200, 500), 255),
                                       ((65, 124), 0)])
def test_bgdiff_gate_fused(vu, shape, thr):
    """the fused, bit-packed gate (vu_bgdiff_gate) against the oracle's bg.py:85-92 restatement: tile seams (120 x 64
    output tiles), image borders, thresholds at the ends of the range, per-frame and shared backgrounds."""
    h, w = shape
    rng = np.random.default_rng(h * 1000 + w + thr)
    n = 3
    bg = rng.integers(0, 256, (n, h, w, 3), dtype=np.uint8)
    frames = np.clip(bg.astype(np.int16) + rng.integers(-20, 21, (n, h, w, 3)), 0, 255).astype(np.uint8)
    hot = rng.random((n, h, w)) < 0.01                     # sparse large differences: isolated dilation footprints
    frames[hot] = 255 - bg[hot]
    frames[:, 0, 0] = 255; bg[:, 0, 0] = 0                 # gray == 255 exactly, in a corner
    frames[:, -1, -1] = 0; bg[:, -1, -1] = 255
    masks = rng.integers(0, 256, (n, h, w), dtype=np.uint8)
    got = vu.ops.bgdiff_gate(torch.from_numpy(frames).cuda(), torch.from_numpy(bg).cuda(), torch.from_numpy(masks).cuda(), thr).cpu().numpy()
    for i in range(n):
        assert np.array_equal(got[i], R.bgdiff_gate(frames[i], bg[i], masks[i], thr)), i
    got1 = vu.ops.bgdiff_gate(torch.from_numpy(frames).cuda(), torch.from_numpy(bg[0]).cuda(), torch.from_numpy(masks).cuda(), thr).cpu().numpy()
    for i in range(n):
        assert np.array_equal(got1[i], R.bgdiff_gate(frames[i], bg[0], masks[i], thr)), i


# ---- temporal ----------------------------------------------------------------------------------

def test_temporal_golden(vu, golden):
    t = golden("temporal")
    U = vu.U
    bg, ma = U.masked_temporal_mean(t["frames"], t["masks"])
    assert np.array_equal(bg, t["mean_bg"]) and np.array_equal(ma, t["mean_mask_always"])
    assert np.array_equal(U.temporal_median(t["frames"]), t["median_even"])
    assert np.array_equal(U.temporal_median(t["frames"][:23]), t["median_odd"])
    assert np.array_equal(U.temporal_median(t["rnd"]), t["median_rnd"])   # 33x47x3: tail path + ragged size


@pytest.mark.parametrize("n", [1, 2, 3, 16, 151, 152, 153, 255, 256, 299, 300, 304, 305, 511, 608, 609, 700])
def test_temporal_median_vs_oracle(vu, n):
    from video_unscreen_b200 import synth
    h, w = 24, 64
    frames = synth.random_clip(n, h, w, seed=n)
    assert np.array_equal(vu.U.temporal_median(frames), R.temporal_median(frames))
    # heavily repeated values (counter wrap / saturation hazards)
    const = np.full((n, h, w, 3), 7, np.uint8)
    const[: n // 3] = 200
    assert np.array_equal(vu.U.temporal_median(const), R.temporal_median(const))
    # two-valued data: for even n the two middle order statistics can be 0 and 255 (longest possible plateau)
    rng = np.random.default_rng(n)
    two = np.where(rng.integers(0, 2, (n, h, w, 3)) > 0, 255, 0).astype(np.uint8)
    two[:, 0] = 0
    two[: n // 2, 0] = 255          # exact half split on row 0
    two[:, 1] = np.where(np.arange(n)[:, None, None] % 2 == 0, 3, 250)
    assert np.array_equal(vu.U.temporal_median(two), R.temporal_median(two))
    # sparse values with gaps of every size
    gaps = (rng.integers(0, 4, (n, h, w, 3)) * rng.integers(1, 80, (1, h, w, 3))).astype(np.uint8)
    assert np.array_equal(vu.U.temporal_median(gaps), R.temporal_median(gaps))


@pytest.mark.parametrize("n", [81, 82, 83, 152, 153, 232, 233, 240, 241, 299, 300, 303, 304, 305, 306, 307, 464, 465, 607, 608,
                               609, 610, 912, 913, 1000, 1217, 2000])
def test_temporal_median_concentrated(vu, n):
    """background-like data (the estimate + windowed search path of vu_median_sad.cuh): static background with small
    temporal noise, occluded for a contiguous run of frames, including backgrounds at the ends of the uint8 range;
    a few elements per warp with wide noise force the fall-back to the full search inside the same warp."""
    rng = np.random.default_rng(1000 + n)
    h, w = 16, 128
    base = rng.integers(0, 256, (h, w, 3)).astype(np.int16)
    base[0] = 0
    base[1] = 255
    base[2] = rng.integers(0, 12, (w, 3))
    base[3] = rng.integers(244, 256, (w, 3))
    frames = base[None] + rng.integers(-6, 7, (n, h, w, 3))
    t0 = n // 5
    frames[t0:t0 + (28 * n) // 100, 4:12, 10:90] = rng.integers(80, 240, ((28 * n) // 100, 8, 80, 3))   # occluder
    frames[:, 8:, ::17] = base[None, 8:, ::17] + rng.integers(-40, 41, (n, h - 8, len(range(0, w, 17)), 3))  # wide noise
    frames[:, 12:, 5] = np.where(rng.integers(0, 2, (n, h - 12, 3)) > 0, base[None, 12:, 5] + 1, base[None, 12:, 5])  # two adjacent values
    frames = np.clip(frames, 0, 255).astype(np.uint8)
    want = R.temporal_median(frames)
    assert np.array_equal(vu.U.temporal_median(frames), want)          # 16-byte aligned: TMA tile kernels
    # the same clip 4 bytes off a 16-byte boundary: direct register kernels (no TMA, no 16-byte requests)
    flat = torch.empty(frames.size + 16, dtype=torch.uint8, device="cuda")
    off = flat[4:4 + frames.size].view(frames.shape)
    off.copy_(torch.from_numpy(frames))
    assert off.data_ptr() % 16 == 4
    assert np.array_equal(vu.ops.temporal_median(off).cpu().numpy(), want)
    # frame size not a multiple of 16 bytes (15 x 100 x 3 = 4500): direct kernels, then the byte tail
    sub = np.ascontiguousarray(frames[:, :15, :100])
    assert np.array_equal(vu.U.temporal_median(sub), R.temporal_median(sub))


def test_temporal_median_properties_full_size(vu):
    """BASELINE config 2 size (300 x 1080p): size-independent properties.
    median of a clip whose frames are a permutation of values is order
    independent; median of [x, x, ..., x] is x; min <= median <= max."""
    n, h, w = 300, 1080, 1920
    g = torch.Generator(device="cuda").manual_seed(0)
    base = torch.randint(0, 256, (h, w, 3), dtype=torch.uint8, device="cuda", generator=g)
    noise = torch.randint(0, 13, (n, h, w, 3), dtype=torch.uint8, device="cuda", generator=g)
    frames = (base.to(torch.int16)[None] + noise.to(torch.int16) - 6).clamp_(0, 255).to(torch.uint8)
    del noise
    med = vu.ops.temporal_median(frames)
    perm = torch.randperm(n, device="cuda", generator=g)
    med2 = vu.ops.temporal_median(frames[perm].contiguous())
    assert torch.equal(med, med2)
    lo = frames.amin(0)
    hi = frames.amax(0)
    assert bool(((med >= lo) & (med <= hi)).all())
    # exact check on a strip against torch's own sort-based order statistics
    strip = frames[:, 500:520].to(torch.int16)
    s, _ = strip.sort(0)
    want = ((s[n // 2 - 1] + s[n // 2]) >> 1).to(torch.uint8)
    assert torch.equal(med[500:520], want)
    del frames
    const = torch.full((n, 8, 64, 3), 77, dtype=torch.uint8, device="cuda")
    assert bool((vu.ops.temporal_median(const) == 77).all())


@pytest.mark.parametrize("mask_op,prior,invert", [(0, None, False), (1, None, False), (0, (40, 70), False), (1, (40, 70), True), (1, (0, 1), False)])
def test_cf_samples_order_exact(vu, mask_op, prior, invert):
    """vu_cf_samples == channel[selection][::len // max] of colorfiltering/agent.py:139-141 for the three channels, plus
    the histogram of the hue samples (:142): same pixels, same order, same stride."""
    rng = np.random.default_rng(11)
    h, w, mx = 135, 240, 1000
    hsv = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
    hsv[..., 0] = rng.integers(30, 90, (h, w))
    mask = rng.integers(0, 256, (h, w), dtype=np.uint8)
    mask[:, :7] = 128                                    # neither < 128 nor > 128
    sel = (mask < 128) if mask_op == 0 else (mask > 128)
    if prior is not None:
        inside = (hsv[..., 0] > prior[0]) & (hsv[..., 0] < prior[1])
        sel = sel & (~inside if invert else inside)
    want = []
    for c in range(3):
        smp = hsv[..., c][sel]
        if len(smp) > mx:
            smp = smp[::len(smp) // mx]
        want.append(smp)
    got, total, hist = vu.ops.cf_samples(torch.from_numpy(hsv).cuda(), torch.from_numpy(mask).cuda(), mask_op, mx, prior=prior, invert=invert)
    assert total == int(sel.sum())
    assert got.shape == (3, len(want[0]))
    for c in range(3):
        assert np.array_equal(got[c], want[c])
    assert np.array_equal(hist, np.histogram(want[0].astype(float), 256, [0, 256])[0])


@pytest.mark.parametrize("sc,th,tw,iters", [(2, 64, 96, 5), (4, 64, 96, 5), (2, 70, 100, 5), (4, 33, 52, 3), (2, 130, 196, 1), (4, 65, 200, 0),
                                            (2, 9, 12, 8), (2, 67, 128, 12)])
def test_trimap_bits_tail(vu, sc, th, tw, iters):
    """vu_trimap_bits (nearest down -> binary cross dilation / erosion -> classification -> snapped bilinear up-scale as tap
    logic) against the oracle's generate_trimap and the ensemble branch of generate_trimap_withbg, tile seams (96 x 64
    working-resolution tiles), borders, grey-valued masks, fuzzy overrides, per-frame flags."""
    h, w = sc * th, sc * tw
    rng = np.random.default_rng(sc * 1000 + th + tw + iters)
    n = 3
    yy, xx = np.mgrid[0:h, 0:w]
    masks = np.zeros((n, h, w), np.uint8)
    for i in range(n):
        blob = (((xx - w * (0.3 + 0.2 * i)) / (w * 0.22)) ** 2 + ((yy - h * 0.5) / (h * 0.38)) ** 2) <= 1
        masks[i][blob] = rng.integers(100, 256, int(blob.sum()))         # grey values either side of 128
        masks[i][rng.random((h, w)) < 0.002] = 255                        # isolated specks
    masks[0, :, :3] = 255; masks[0, :2, :] = 255                          # touching the borders
    masks[1, -1, :] = 255; masks[1, :, -1] = 200
    long_side = max(th, tw)
    want = np.stack([R.generate_trimap(masks[i], long_side, 3, iters) for i in range(n)])
    got = vu.ops.trimap_bits(torch.from_numpy(masks).cuda(), th, tw, iters).cpu().numpy()
    assert np.array_equal(got, want)
    # ensemble branch (trimap/agent.py:96-100): fuzzy pixels cleared before, set to 128 after; flags pick the frames
    fuzzy = ((rng.random((n, h, w)) < 0.05) & (masks > 0)).astype(np.uint8)
    flags = np.array([0, 1, 0], np.uint8)
    want2 = []
    for i in range(n):
        if flags[i] == 0:
            m = masks[i].copy()
            m[fuzzy[i] > 0] = 0
            t = R.generate_trimap(m, long_side, 3, iters)
            t[fuzzy[i] > 0] = 128
        else:
            t = R.generate_trimap(masks[i], long_side, 3, iters)
        want2.append(t)
    got2 = vu.ops.trimap_bits(torch.from_numpy(masks).cuda(), th, tw, iters, torch.from_numpy(fuzzy).cuda(), torch.from_numpy(flags).cuda()).cpu().numpy()
    assert np.array_equal(got2, np.stack(want2))


@pytest.mark.parametrize("sc,th,tw", [(2, 1, 32), (2, 7, 64), (4, 13, 32), (2, 40, 1024), (4, 200, 96), (2, 150, 160), (4, 11, 992), (2, 97, 960)])
def test_trimap_bits_marching(vu, sc, th, tw):
    """vu_trimap_bits_packed at working widths of whole 32-pixel words and the reference's 5 passes: the marching kernel
    (trimap_bits_march_kernel: one warp per band of rows, 1 .. 32 word columns, bands shorter than their halo, one-row
    images, several frames) against the oracle's generate_trimap and the ensemble branch of generate_trimap_withbg."""
    h, w = sc * th, sc * tw
    rng = np.random.default_rng(sc * 7919 + th * 31 + tw)
    n = 3
    masks = np.zeros((n, h, w), np.uint8)
    yy, xx = np.mgrid[0:h, 0:w]
    for i in range(n):
        blob = (((xx - w * (0.25 + 0.25 * i)) / (w * 0.2)) ** 2 + ((yy - h * 0.5) / (h * 0.4)) ** 2) <= 1
        masks[i][blob] = rng.integers(100, 256, int(blob.sum()))
        masks[i][rng.random((h, w)) < 0.01] = 255
        masks[i][rng.random((h, w)) < 0.01] = 0
    masks[0, :, : 2 * sc] = 255; masks[0, : 2 * sc, :] = 255              # touching the borders (word 0 / the last word)
    masks[1, -sc:, :] = 255; masks[1, :, -sc:] = 200
    masks[2, :, w // 2 - sc: w // 2 + sc] = 255                           # a bar across a word seam
    fuzzy = ((rng.random((n, h, w)) < 0.05) & (masks > 0)).astype(np.uint8)
    flags = np.array([0, 1, 0], np.uint8)
    long_side = max(th, tw)
    want, want_plain = [], []
    for i in range(n):
        plain = R.generate_trimap(masks[i], long_side, 3, 5)
        want_plain.append(plain)
        if flags[i] == 0:
            m = masks[i].copy()
            m[fuzzy[i] > 0] = 0
            t = R.generate_trimap(m, long_side, 3, 5)
            t[fuzzy[i] > 0] = 128
        else:
            t = plain
        want.append(t)
    mb = np.packbits((masks[:, ::sc, ::sc] >= 128).astype(np.uint8), axis=-1, bitorder="little")
    fzb = np.packbits(fuzzy, axis=-1, bitorder="little")
    ops = vu.ops
    got_plain = ops.trimap_bits_packed(torch.from_numpy(mb).cuda(), None, None, h, w, th, tw, 5).cpu().numpy()
    assert np.array_equal(got_plain, np.stack(want_plain))
    got = ops.trimap_bits_packed(torch.from_numpy(mb).cuda(), torch.from_numpy(fzb).cuda(), torch.from_numpy(flags).cuda(), h, w, th, tw, 5).cpu().numpy()
    assert np.array_equal(got, np.stack(want))


@pytest.mark.parametrize("sc,sh,sw", [(2, 135, 240), (4, 90, 160), (2, 7, 12), (4, 5, 6), (2, 33, 100), (4, 67, 34)])
def test_resize_up_exact_scales(vu, sc, sh, sw):
    """vu_resize_up_u8 on exact 2x / 4x scales (the constant-weight kernel) against the cv2 model: random grey maps (every
    phase, every border), plus the early-out frames copied from the alternative source."""
    rng = np.random.default_rng(sc * 100 + sh + sw)
    n = 3
    src = rng.integers(0, 256, (n, sh, sw), dtype=np.uint8)
    dh, dw = sc * sh, sc * sw
    want = np.stack([M.resize_linear(x, dw, dh) for x in src])
    got = host(vu.ops.resize_up(dev(src), dh, dw))
    assert np.array_equal(got, want)
    alt = rng.integers(0, 256, (n, dh, dw), dtype=np.uint8)
    flags = np.array([0, 2, 1], np.uint8)
    got = host(vu.ops.resize_up(dev(src), dh, dw, alt_src=dev(alt), alt_flags=dev(flags)))
    assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], alt[1]) and np.array_equal(got[2], alt[2])


SHIFTS = [(3, -2), (0.5, 0.5), (0, 0), (-7.3, 4.9), (12.015625, -0.984375), (1e-3, 33.333), (-100, 2), (0.484375, 0.515625), (5.7, 200),
          (-0.015, -0.016), (1e-30, -1e-30)]


@pytest.mark.parametrize("shape", [(64, 80, 3), (64, 80), (61, 83, 3), (45, 37), (135, 240, 3), (70, 496, 3), (33, 1024)])
def test_shift_fg(vu, shape):
    """shift_fg (imgprocess.py:55-64) through both kernels -- the TMA tile kernel (rows of a multiple of 16 bytes) and the
    generic one (anything else) -- against the fixed-point warpAffine model: bit-exact, every sub-pixel phase class,
    shifts that leave the frame, clips (frames must not leak into each other)."""
    rng = np.random.default_rng(sum(shape))
    clip = rng.integers(0, 256, (3,) + shape, dtype=np.uint8)
    ch = 3 if len(shape) == 3 else 1
    for dx, dy in SHIFTS:
        want = np.stack([M.warp_translate(f, dx, dy) for f in clip])
        got = host(vu.ops.shift(dev(clip), dx, dy, ch))
        assert np.array_equal(got, want), (shape, dx, dy, int((got != want).sum()))
    img = clip[0]
    assert np.array_equal(vu.U.shift_fg(img, dx=2.25, dy=-3.75), M.warp_translate(img, 2.25, -3.75))


@pytest.mark.parametrize("shape", [(64, 80, 3), (64, 80), (61, 83, 3), (45, 37), (135, 240, 3), (40, 700), (100, 130, 3)])
def test_rescale_fg(vu, shape):
    """rescale_fg (imgprocess.py:40-52) against the float bicubic model: bit-exact (same float32 operation order), for
    the script's factor 1.2, the default 1.1, and factors whose taps reach over the border (1.0, 1.01) or skip rows (3.7)."""
    rng = np.random.default_rng(sum(shape) + 1)
    clip = rng.integers(0, 256, (2,) + shape, dtype=np.uint8)
    ch = 3 if len(shape) == 3 else 1
    for f in (1.2, 1.1, 1.0, 1.01, 1.5, 2.0, 3.7):
        want = np.stack([M.resize_cubic_crop(x, f) for x in clip])
        got = host(vu.ops.rescale_cubic(dev(clip), f, ch))
        assert np.array_equal(got, want), (shape, f, int((got != want).sum()))
    assert np.array_equal(vu.U.rescale_fg(clip[0], 1.2), M.resize_cubic_crop(clip[0], 1.2))


def test_replace_with_geometry(vu):
    """replace.py:69-76 end to end: shift + rescale of foreground and (3-channel and single-channel) mask, then the
    float64 blend; every stage is bit-exact against the oracle, so the composite is too."""
    from video_unscreen_b200 import clip as C
    rng = np.random.default_rng(9)
    n, h, w = 3, 96, 160
    fg = rng.integers(0, 256, (n, h, w, 3), dtype=np.uint8)
    a = rng.integers(0, 256, (n, h, w), dtype=np.uint8)
    a3 = np.repeat(a[..., None], 3, axis=3)
    bg = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
    for dx, dy, sc in [(3, -2, 1.2), (0.5, 0.5, 1.2), (-4.3, 7.9, 1.1)]:
        want = np.stack([R.replace_frame(fg[i], a3[i], bg, dx, dy, sc) for i in range(n)])
        assert np.array_equal(host(C.replace_clip(dev(fg), dev(a3), dev(bg), dx, dy, sc)), want)
        assert np.array_equal(host(C.replace_clip(dev(fg), dev(a), dev(bg), dx, dy, sc)), want)


def test_geometry_golden(vu, golden):
    """shift_fg / rescale_fg / the replace.py:69-76 frame against outputs of the unmodified reference (tests/golden/
    geometry.npz): shift bit-exact; rescale within the tie tolerance documented in oracle/cvmodel.py."""
    from video_unscreen_b200 import clip as C
    g = golden("geometry")
    fg, m3, bg = g["fg"], g["mask3"], g["bg"]
    for i, (dx, dy) in enumerate(g["shifts"]):
        assert np.array_equal(vu.U.shift_fg(fg, dx=dx, dy=dy), g[f"shift_fg_{i}"]), (dx, dy)
        assert np.array_equal(vu.U.shift_fg(m3[..., 0], dx=dx, dy=dy), g[f"shift_mask_{i}"]), (dx, dy)
    for tag, sc in (("12", 1.2), ("11", 1.1)):
        for mine, ref in ((vu.U.rescale_fg(fg, sc), g[f"rescale_fg_{tag}"]), (vu.U.rescale_fg(m3[..., 0], sc), g[f"rescale_mask_{tag}"])):
            d = np.abs(mine.astype(int) - ref.astype(int))
            assert d.max() <= 1 and (d > 0).mean() <= 1e-4
    got = host(C.replace_clip(dev(fg[None]), dev(m3[None]), dev(bg), 3, -2, 1.2))[0]
    d = np.abs(got.astype(int) - g["replace_frame"].astype(int))
    assert d.max() <= 2 and (d > 0).mean() <= 1e-3


@pytest.mark.parametrize("h,w,L", [(108, 192, 96), (216, 384, 96), (150, 110, 60), (96, 160, 160), (270, 480, 240)])
def test_color_correct(vu, h, w, L):
    """color_correct (imgprocess.py:263-300) against the oracle (itself bit-exact against the live reference in
    tests/test_oracle_vs_reference.py): bit-exact, single images through the reference-shaped function and a clip through
    the batched op; working resolutions that are the frame size, half of it, and a non-integer ratio; mattes that are
    empty (no iteration) and a frame of one single colour (0 / 0: the reference's NaN casts to 0)."""
    from video_unscreen_b200 import synth
    n = 3
    frames, segs = synth.green_clip(n, h, w, seed=h + L)
    rng = np.random.default_rng(w)
    alphas = np.stack([np.minimum(np.where(rng.random((h, w)) < 0.3, rng.integers(0, 256, (h, w)), 255).astype(np.uint8), segs[i]) for i in range(n)])
    alphas[2] = 0
    th, tw = R.get_target_size(h, w, L)
    for col in ((60, 200, 40), (200, 30, 30)):
        c = np.array(col, np.uint8)
        want = np.stack([R.color_correct(frames[i], alphas[i], c, target_long_side=L) for i in range(n)])
        got = host(vu.ops.color_correct(dev(frames), dev(alphas), c, th, tw))
        assert np.array_equal(got, want), (col, int((got != want).sum()))
        assert np.array_equal(vu.U.color_correct(frames[0], alphas[0], c, target_long_side=L), want[0])
    flat = np.full((h, w, 3), 77, np.uint8)
    a = np.full((h, w), 200, np.uint8)
    c = np.array((60, 200, 40), np.uint8)
    assert np.array_equal(vu.U.color_correct(flat, a, c, target_long_side=L), R.color_correct(flat, a, c, target_long_side=L))


def test_color_correct_golden(vu, golden):
    """color_correct against outputs of the unmodified reference (tests/golden/geometry.npz): bit-exact; the 1/2 working
    resolution takes the fused down-scale kernel, the others the resize + vu_color_correct path."""
    g = golden("geometry")
    for ci, col in enumerate(g["cc_colors"]):
        for L in g["cc_long_sides"]:
            for i in range(2):
                got = vu.U.color_correct(g["cc_frames"][i], g["cc_alpha"][i], col, target_long_side=int(L))
                assert np.array_equal(got, g[f"cc_{ci}_{int(L)}_{i}"]), (ci, int(L), i)


@pytest.mark.parametrize("n,h,w", [(7, 40, 64), (24, 33, 272), (5, 16, 128), (12, 50, 400), (9, 21, 16)])
def test_masked_mean_fused_dilation(vu, n, h, w):
    """the masked temporal mean with dilate_mask(mask, 3, 2) fused in as bit-plane logic (vu_masked_temporal_mean_dilate32)
    against the oracle (dilate, then mean) and against the unfused kernels: grey masks with values around both thresholds
    (250, 255), features on tile borders and image borders."""
    rng = np.random.default_rng(n * h + w)
    frames = rng.integers(0, 256, (n, h, w, 3), dtype=np.uint8)
    masks = rng.choice(np.array([0, 0, 0, 0, 0, 0, 0, 120, 249, 250, 254, 255, 255], np.uint8), size=(n, h, w))
    masks[:, :, ::37] = 0
    masks[:, 0, :] = np.where(rng.random((n, w)) < 0.3, 255, 0)
    masks[:, :, w - 1] = np.where(rng.random((n, h)) < 0.3, 255, 0)
    masks[0] = 255
    want_bg, want_always = R.masked_temporal_mean(frames, masks, min_count=2)
    bg, always = vu.ops.masked_temporal_mean_raw(dev(frames), dev(masks), 3, 2, 2)
    assert np.array_equal(host(bg), want_bg) and np.array_equal(host(always), want_always)
    bg2, always2 = vu.ops.masked_temporal_mean(dev(frames), vu.ops.dilate(dev(masks), 3, 2), 2)
    assert np.array_equal(host(bg), host(bg2)) and np.array_equal(host(always), host(always2))


def test_replace_geometry_full_size(vu):
    """shift_fg / rescale_fg at BASELINE config 4's frame size (1080p): identities (a zero shift and a unit scale return
    the clip), an integer shift and its inverse restore everything that stayed inside the frame, and one whole frame of
    each against the oracle."""
    from video_unscreen_b200 import synth
    frames, _ = synth.green_clip(3, 1080, 1920, seed=21)
    d = dev(frames)
    assert torch.equal(vu.ops.shift(d, 0, 0, 3), d)
    assert torch.equal(vu.ops.rescale_cubic(d, 1.0, 3), d)
    back = vu.ops.shift(vu.ops.shift(d, 37, -21, 3), -37, 21, 3)
    # dx = 37 moves the content right, dy = -21 moves it up: the rows below 21 and the columns from 1920 - 37 on left the frame
    assert torch.equal(back[:, 21:, : 1920 - 37], d[:, 21:, : 1920 - 37])
    assert not bool(back[:, :21].any()) and not bool(back[:, :, 1920 - 37:].any())          # ... and came back as border
    assert np.array_equal(host(vu.ops.shift(d[:1], 0.5, 0.5, 3))[0], M.warp_translate(frames[0], 0.5, 0.5))
    assert np.array_equal(host(vu.ops.rescale_cubic(d[1:2], 1.2, 3))[0], M.resize_cubic_crop(frames[1], 1.2))


@pytest.mark.parametrize("h,w", [(1080, 1920), (2160, 3840)])
def test_color_correct_full_size(vu, h, w):
    """color_correct at the two BASELINE frame sizes (working resolution 540 x 960: the fused 2x and 4x down-scale
    kernels) against the oracle, one frame each, plus the property that the result never exceeds alpha."""
    from video_unscreen_b200 import synth
    frames, segs = synth.green_clip(2, h, w, seed=h)
    rng = np.random.default_rng(h)
    alpha = np.minimum(segs, rng.integers(100, 256, segs.shape).astype(np.uint8))
    col = np.array([60, 200, 40], np.uint8)
    th, tw = R.get_target_size(h, w, 960)
    got = host(vu.ops.color_correct(dev(frames), dev(alpha), col, th, tw))
    assert np.array_equal(got[1], R.color_correct(frames[1], alpha[1], col))
    assert bool((got <= alpha).all())


@pytest.mark.parametrize("i", range(5))
def test_background_agent_golden(vu, golden, i):
    """SURVEY 8f rank 4: BackgroundAgent.forward 'pcov' and 'mean' on the device: bit-exact against the oracle; against the
    reference's goldens 'pcov' bit-exact, 'mean' within the HSV2BGR tolerance (<= 2 LSB after the final resize)."""
    from video_unscreen_b200.unscreen.bgmodel import BackgroundAgent
    g = golden("bgmodel")
    h, w, L, kind = (int(v) for v in g["cases"][i])
    img, m = g[f"img_{i}"], g[f"mask_{i}"]
    ag = BackgroundAgent(input_long_side=L)
    got = ag.forward(img, m, "pcov")
    assert np.array_equal(got, R.background_forward(img, m, "pcov", input_long_side=L))
    assert np.array_equal(got, g[f"pcov_{i}"])
    got = ag.forward(img, m, "mean")
    assert np.array_equal(got, R.background_forward(img, m, "mean", input_long_side=L))
    assert maxdiff(got, g[f"mean_{i}"]) <= 2
    # early-outs, error behaviour, device tensors in -> device tensors out
    assert ag.forward(img, np.zeros_like(m), "pcov") is img
    z = ag.forward(img, np.full_like(m, 255), "mean")
    assert z.dtype == np.float64 and z.shape == img.shape and not z.any()
    with pytest.raises(NameError):
        ag.forward(img, m, "telea")
    t = ag.forward(dev(img), dev(m), "pcov")
    assert t.is_cuda and np.array_equal(host(t), g[f"pcov_{i}"])
    ag3 = BackgroundAgent(input_long_side=L, dilation_ksize=3, dilation_iters=2, pcov_ksize=3)
    assert np.array_equal(ag3.forward(img, m, "pcov"),
                          R.background_forward(img, m, "pcov", input_long_side=L, dilation_ksize=3, dilation_iters=2, pcov_ksize=3))


@pytest.mark.parametrize("i", range(5))
def test_regionfill_golden(vu, golden, i):
    """SURVEY 8f rank 4: regionfill (utils/region_fill.py) and BackgroundAgent.forward(method='rf').  The reference solves
    the Laplace system directly (scipy spsolve), the device by conjugate gradients to a relative residual of 1e-10: the
    tolerance is |difference| <= 1e-5 grey levels on the float result; after the reference's truncation to uint8 that is
    <= 1 LSB on at most 1e-4 of the pixels (values that sit on an integer).  'rf' then ends in HSV2BGR: <= 2 LSB after the
    final resize against the reference (the scalar tail of cv2's HSV2BGR, as for 'mean'), near-exact against the oracle."""
    from video_unscreen_b200.unscreen.bgmodel import BackgroundAgent
    g = golden("regionfill")
    h, w, L, kind = (int(v) for v in g["cases"][i])
    img, m = g[f"img_{i}"], g[f"mask_{i}"]
    plane = np.ascontiguousarray(img[:, :, i % 3])
    for f in (1.0, 0.5):
        want = g[f"fill_{i}_{int(f * 10)}"]
        got = vu.U.regionfill(plane, m > 0, f)
        assert got.dtype == np.float64 and got.shape == want.shape
        assert np.abs(got - want).max() <= 1e-5, (f, np.abs(got - want).max())
        flips = got.astype(np.uint8) != want.astype(np.uint8)
        assert flips.mean() <= 1e-4 and maxdiff(got.astype(np.uint8), want.astype(np.uint8)) <= 1
        assert np.array_equal(got[m == 0], plane[m == 0].astype(np.float64))
    # uint8 0 / 255 mask (bg.py:79), three planes in one solve (CUDA tensors in -> CUDA tensor out), empty mask
    planes = dev(np.ascontiguousarray(img.transpose(2, 0, 1)))
    got3 = vu.U.regionfill(planes, dev(m), 1.0)
    assert got3.is_cuda and got3.dtype == torch.float64
    assert np.abs(host(got3)[i % 3] - g[f"fill_{i}_10"]).max() <= 1e-5
    assert np.array_equal(vu.U.regionfill(plane, np.zeros_like(m)), plane)
    # the agent
    ag = BackgroundAgent(input_long_side=L)
    got = ag.forward(img, m, "rf")
    assert got.dtype == np.uint8 and got.shape == img.shape
    assert maxdiff(got, g[f"rf_{i}"]) <= 2
    orc = R.background_forward(img, m, "rf", input_long_side=L)
    assert maxdiff(got, orc) <= 1 and (got != orc).mean() <= 1e-3, ((got != orc).mean(), maxdiff(got, orc))
    assert BackgroundAgent().forward(img, m).shape == img.shape          # 'rf' is the default method (:159)


@pytest.mark.parametrize("i", range(6))
def test_remove_invalid_objects_golden(vu, golden, i):
    """SURVEY 8f rank 2: remove_invalid_objects on the device (union-find labelling of both classes, nesting tree, local
    boundary counts, one CTA per frame for the tree) against the reference's goldens and the oracle, bit-exact; the three
    configurations as one batched call; a table that is too small is redone"""
    import os, sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
    from make_golden import OBJ_CFGS
    g = golden("objects")
    a, seg = g[f"alpha_{i}"], g[f"seg_{i}"]
    for c, cfg in enumerate(OBJ_CFGS):
        assert np.array_equal(vu.U.remove_invalid_objects(cfg, a), g[f"self_{i}_{c}"]), c
        assert np.array_equal(vu.U.remove_invalid_objects(cfg, a, seg), g[f"seg_{i}_{c}"]), c
    cfg = OBJ_CFGS[1]
    clip_a = np.stack([a, np.zeros_like(a), np.full_like(a, 255), a[::-1].copy()])
    clip_s = np.stack([seg, seg, seg, seg[::-1].copy()])
    got = vu.U.remove_invalid_objects(cfg, clip_a, clip_s)
    for k in range(4):
        assert np.array_equal(got[k], R.remove_invalid_objects(cfg, clip_a[k], clip_s[k])), k
    assert np.array_equal(vu.U.remove_invalid_objects(cfg, a, seg, max_objects=4), g[f"seg_{i}_1"])
    t = vu.U.remove_invalid_objects(cfg, dev(a), dev(seg))
    assert t.is_cuda and np.array_equal(host(t), g[f"seg_{i}_1"])


def test_remove_invalid_objects_shapes(vu):
    """hand-made nesting: ring with an island that has its own hole, 1-pixel-wide parts, objects on the image border,
    diagonal contacts (8-connected foreground / 4-connected background), areas either side of 100"""
    import os, sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
    from make_golden import OBJ_CFGS
    from test_oracle_objects_fast import handmade_objects
    a, seg = handmade_objects()
    for cfg in OBJ_CFGS:
        for s in (None, seg):
            assert np.array_equal(vu.U.remove_invalid_objects(cfg, a, s), R.remove_invalid_objects(cfg, a, s)), (cfg, s is None)
    rng = np.random.default_rng(3)
    for trial in range(6):         # salt and pepper: thousands of components
        x = (rng.random((72, 100)) < (0.35 + 0.08 * trial)).astype(np.uint8) * 255
        cfg = {'objectremoval': {'score_map_center': {'landscape': [0.5, 0.5], 'portrait': [0.6, 0.5]}, 'saliency_thr': 1e-7, 'consensus_thr': 0.1}}
        assert np.array_equal(vu.U.remove_invalid_objects(cfg, x, max_objects=256), R.remove_invalid_objects(cfg, x)), trial


@pytest.mark.parametrize("h,w", [(33, 47), (5, 3), (1, 1), (35, 64)])
def test_compositing_odd_sizes_and_views(vu, h, w):
    """ADVICE r1: frames whose pixel count is not a multiple of 4, and unaligned views, go to the one-pixel-per-thread
    kernels instead of raising; a background of the wrong shape raises instead of wrapping around"""
    rng = np.random.default_rng(h * 100 + w)
    fr = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
    bg = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
    al = rng.integers(0, 256, (h, w), dtype=np.uint8)
    al[rng.random((h, w)) < 0.3] = 0
    assert np.array_equal(vu.U.get_fg(fr, al, bg), R.get_fg(fr, al, bg))
    assert np.array_equal(vu.U.get_fg(fr, al, bg, patch="eq0"), R.get_fg(fr, al, R.patch_bg(bg, fr, al, "eq0")))
    assert np.array_equal(vu.U.get_bg(al, bg), R.get_bg(al, bg))
    assert np.array_equal(vu.U.get_fg_naive(fr, al), R.get_fg_naive(fr, al))
    assert np.array_equal(vu.U.fuse_fgbg(fr, bg, al), R.fuse_fgbg(fr, bg, al))
    assert np.array_equal(vu.U.replace_blend(fr, al, bg), R.replace_blend(fr, al, bg))
    assert np.array_equal(vu.U.replace_blend(fr, np.stack([al] * 3, -1), bg), R.replace_blend(fr, al, bg))
    assert np.array_equal(vu.U.composite_fgbg(fr, al, bg), R.composite_fgbg(fr, al, bg))
    assert np.array_equal(vu.U.fuse_bg(fr, bg, 0.1), R.fuse_bg(fr, bg, 0.1))
    assert np.array_equal(vu.U.bgdiff_gate(fr, bg, al, 25), R.bgdiff_gate(fr, bg, al, 25))
    # an unaligned view: one byte into a larger buffer
    buf = torch.zeros(h * w * 3 + 8, dtype=torch.uint8, device="cuda")
    view = buf[1:1 + h * w * 3].view(h, w, 3)
    view.copy_(dev(fr))
    got = vu.ops.get_fg(view, dev(al), dev(bg))
    assert np.array_equal(host(got), R.get_fg(fr, al, bg))
    if h > 1:
        with pytest.raises(ValueError):
            vu.ops.get_fg(dev(fr), dev(al), dev(bg[: h - 1]))
        with pytest.raises(ValueError):
            vu.ops.blend(3, dev(fr), dev(al), dev(bg[:, : w - 1].copy()) if w > 1 else dev(bg[: h - 1]))


@pytest.mark.parametrize("k,n", [(9, 2), (11, 1), (15, 1), (7, 45), (5, 70), (4, 80)])
def test_morphology_large(vu, k, n):
    """ADVICE r1: structuring elements above 7x7 and iteration counts whose halo does not fit one launch's shared memory
    (several launches through a scratch image) instead of VU_ERR_UNSUPPORTED"""
    rng = np.random.default_rng(k * 100 + n)
    m = rng.integers(0, 256, (2, 150, 170), dtype=np.uint8)
    m[0, 40:110, 50:120] = 0
    m[1, 10:60, 10:90] = 255
    for op, ref in ((vu.ops.dilate, M.dilate), (vu.ops.erode, M.erode)):
        got = host(op(dev(m), k, n))
        assert np.array_equal(got, np.stack([ref(x, k, n) for x in m])), (k, n)
