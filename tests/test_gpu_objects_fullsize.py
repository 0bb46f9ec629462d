"""remove_invalid_objects on the device at 1080p and 4K, bit-exact against the whole-array contour model
(oracle/refport.py:remove_invalid_objects_fast, itself checked against the per-contour closed form in
tests/test_oracle_objects_fast.py): millions of pixels across thousands of CTAs for the lock-free union-find, tens of
thousands of contours (more than the default table: the redo path), one diagonal-only component around a million holes,
a frame-crossing 1-px path, nesting hundreds of levels deep, per-frame workspace slices of a batched clip, and
green_clip with tracked and untracked frames.  Every case first asserts that no contour's saliency lies within 1e-9
(relative) of a threshold, where the device's float64 atomic sums and the model's sums could disagree."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

from oracle import refport as R  # noqa: E402
from test_oracle_objects_fast import OBJ_CFGS, blobby, checker, rings, salt, segmask_for, serpentine  # noqa: E402

HD, UHD = (1080, 1920), (2160, 3840)
MARGIN = 1e-9


@pytest.fixture(scope="module")
def U():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import video_unscreen_b200.unscreen.utils as U
    return U


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def model(cfg, a, seg):
    """the model's output; refuses a case a summation order could decide"""
    want, rec = R.remove_invalid_objects_fast(cfg, a, seg, return_records=True)
    assert R.decision_margin(rec) > MARGIN, "a saliency sits on a threshold: pick another seed"
    return want, rec


def check(U, cfg, a, seg=None):
    want, rec = model(cfg, a, seg)
    got = U.remove_invalid_objects(cfg, a, seg)
    if not np.array_equal(got, want):
        bad = np.argwhere(got != want)
        raise AssertionError(f"{bad.shape[0]} pixels differ, first at {bad[:5].tolist()}; {len(rec['area'])} contours")
    return want, rec


def squares(h, w):
    """11 x 11 squares (contour area exactly 100: not too small), 10 x 10 (81: too small) and 11 x 12 (110) on a grid, and bars
    along every border and in every corner"""
    a = np.zeros((h, w), np.uint8)
    for k, y in enumerate(range(40, h - 60, 60)):
        for j, x in enumerate(range(40, w - 60, 60)):
            s = [(11, 11), (10, 10), (11, 12)][(k + j) % 3]
            a[y:y + s[0], x:x + s[1]] = 255
    a[0:20, 300:700] = 180
    a[h - 15:h, 200:900] = 180
    a[100:400, 0:12] = 180
    a[500:800, w - 30:w] = 180
    for y, x in ((0, 0), (0, w - 25), (h - 25, 0), (h - 25, w - 25)):
        a[y:y + 25, x:x + 25] = 250
    a[h // 2 - 5:h // 2 + 5, w // 2 - 5:w // 2 + 5] = 0      # a hole in no object: stays 0
    return a


@pytest.mark.parametrize("size", [HD, UHD], ids=["1080p", "4k"])
def test_blobby(U, size):
    """grey-valued blobby mattes (every non-zero value is foreground): holes, islands in holes, contour areas around
    100, with and without a segmentation mask, all three configurations"""
    h, w = size
    rng = np.random.default_rng(h)
    a = blobby(rng, h, w, 3.0, 0.6)
    a[rng.random((h, w)) < 0.005] = 200
    seg = segmask_for(np.random.default_rng(1), h, w)
    cfgs = OBJ_CFGS if h == HD[0] else OBJ_CFGS[1:2]
    for cfg in cfgs:
        for s in (None, seg):
            want, rec = check(U, cfg, a, s)
    assert 0 < np.count_nonzero(want) < np.count_nonzero(a)          # removes some objects, keeps others


@pytest.mark.parametrize("size", [HD, UHD], ids=["1080p", "4k"])
def test_percolation(U, size):
    """random sites at density 0.41: 8-connected foreground and its 4-connected background both near their percolation
    thresholds, frame-spanning components with tortuous borders, tens of thousands of contours (the table is redone)"""
    h, w = size
    a = salt(np.random.default_rng(7 + h), h, w, 0.41)
    want, rec = check(U, OBJ_CFGS[1], a)
    assert len(rec["area"]) > 16384
    check(U, OBJ_CFGS[2], a, segmask_for(np.random.default_rng(2), h, w))


def test_checkerboard(U):
    """one diagonal-only foreground component around about a million one-pixel holes"""
    h, w = HD
    a = checker(h, w)
    want, rec = check(U, OBJ_CFGS[1], a)
    assert len(rec["area"]) > 1_000_000 and np.array_equal(want, a)
    seg = np.zeros_like(a)
    seg[:, : w // 3] = 255
    check(U, OBJ_CFGS[2], a, seg)


@pytest.mark.parametrize("size", [HD, UHD], ids=["1080p", "4k"])
def test_serpentine(U, size):
    """a single 1-px path through every other row, with a filled square on its end: the component is kept only if the
    union-find joins the whole path into one set"""
    h, w = size
    a = serpentine(h, w, 2, 40)
    want, rec = check(U, OBJ_CFGS[2], a)
    assert len(rec["area"]) == 1 and np.array_equal(want, a)
    check(U, OBJ_CFGS[2], a.T.copy())


@pytest.mark.parametrize("levels", [64, 65, 66, 530])
def test_nesting_depth(U, levels):
    """concentric 1-px rings on a 2-px pitch, nested 64, 65, 66 and 530 levels deep"""
    h, w = HD
    a = rings(h, w, levels)
    seg = np.zeros_like(a)
    seg[:, : w // 2 + 7] = 255
    for cfg in (OBJ_CFGS[0], OBJ_CFGS[2]):
        want, rec = check(U, cfg, a, seg)
        assert rec["depth"].max() == levels
    check(U, OBJ_CFGS[1], a)


def test_nesting_depth_4k(U):
    """a thousand nested levels, off centre; only a band of middle levels is valid (the outer ones fail consensus, the
    inner ones saliency), so the output is the rings inside that band"""
    h, w = UHD
    a = rings(h, w, 1000, 1070, 1500)
    yy, xx = np.indices((h, w))
    seg = ((yy - 1070) ** 2 + (xx - 1500) ** 2 < 450 ** 2).astype(np.uint8) * 255
    cfg = {'objectremoval': {'score_map_center': {'landscape': [0.5, 0.5], 'portrait': [0.6, 0.5]}, 'saliency_thr': 0.05,
                             'consensus_thr': 0.5}}
    want, rec = check(U, cfg, a, seg)
    assert rec["depth"].max() == 1000 and 0 < np.count_nonzero(want) < np.count_nonzero(a)


def test_degenerate_and_border_frames(U):
    """all 0, all 255, objects on every border and in every corner, squares either side of contour area 100; a portrait
    frame (the other score-map centre)"""
    h, w = HD
    for a in (np.zeros((h, w), np.uint8), np.full((h, w), 255, np.uint8)):
        for cfg in OBJ_CFGS:
            check(U, cfg, a)
    a = squares(h, w)
    want, rec = check(U, OBJ_CFGS[1], a)
    assert rec["valid"][rec["area"] == 100].sum() > 100
    check(U, OBJ_CFGS[0], a, segmask_for(np.random.default_rng(3), h, w))
    p = blobby(np.random.default_rng(9), w, h, 3.0, 0.6)             # 1920 x 1080
    for cfg in OBJ_CFGS:
        check(U, cfg, p, segmask_for(np.random.default_rng(4), w, h))


def test_batched_clip(U):
    """mixed frames with per-frame segmasks in one call (per-frame workspace slices and statuses, one frame over the
    default table); the same call twice gives identical output"""
    h, w = HD
    rng = np.random.default_rng(11)
    clip = np.stack([blobby(rng, h, w, 3.0, 0.6), salt(rng, h, w, 0.41), rings(h, w, 66), np.zeros((h, w), np.uint8),
                     squares(h, w), checker(h, w, 1)])
    segs = np.stack([segmask_for(rng, h, w) for _ in range(len(clip))])
    cfg = OBJ_CFGS[2]
    a_d, s_d = dev(clip), dev(segs)
    got = U.remove_invalid_objects(cfg, a_d, s_d)
    again = U.remove_invalid_objects(cfg, a_d, s_d)
    assert torch.equal(got, again)
    got = got.cpu().numpy()
    for k in range(len(clip)):
        want, _ = model(cfg, clip[k], segs[k])
        assert np.array_equal(got[k], want), k


def test_green_clip_tracked_frames(golden):
    """green.py:106-109: a tracked frame is scored against its own colour-filter alpha, an untracked one against its
    segmentation mask.  A person-coloured square outside the segmentation masks: the untracked frames clear it, the
    tracked ones keep it; alpha, trimap, fg and bg of every frame equal the per-frame oracle chain"""
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from test_oracle_golden import cf_tables
    from video_unscreen_b200 import clip, synth
    from video_unscreen_b200.unscreen.colorfiltering import ColorFilteringAgent
    from video_unscreen_b200.unscreen.trimap import TrimapAgent
    n, (h, w), L = 4, HD, 960
    frames, segs = synth.green_clip(n, h, w, seed=41)
    box = (slice(120, 270), slice(150, 300))
    frames[:, box[0], box[1]] = np.array(synth.PERSON, np.uint8)
    assert not segs[:, box[0], box[1]].any()
    lb, lf, bgh = cf_tables(golden("colorfilter"), "x2")
    cf = ColorFilteringAgent(input_long_side=L)
    cf.set_tables(lb, lf, bgh)
    ta = TrimapAgent(input_long_side=L)
    col = cf.bg_color_bgr()
    cfg = OBJ_CFGS[2]
    tracked = [False, True, True, False]
    outs = [clip.green_clip(dev(frames), dev(segs), cf, ta, chunk=3, remove_objects=cfg, tracked=t)
            for t in (tracked, torch.tensor(tracked, device="cuda"))]
    for a, b in zip(*outs):
        assert torch.equal(a, b)
    alpha, tri, fg, bgo = (t.cpu().numpy() for t in outs[0])
    for i in range(n):
        a_cf, _, _ = R.cf_forward_predict(frames[i], segs[i], lb, lf, bgh, L)
        a_o = R.remove_invalid_objects(cfg, a_cf, None if tracked[i] else segs[i])
        assert np.array_equal(alpha[i], a_o), i
        assert np.array_equal(tri[i], R.generate_trimap_withbg(a_o, frames[i], col, L)), i
        patched = R.patch_bg(np.broadcast_to(col, frames[i].shape), frames[i], a_o, "lt128")
        assert np.array_equal(bgo[i], patched) and np.array_equal(fg[i], R.get_fg(frames[i], a_o, patched)), i
        kept = np.count_nonzero(alpha[i][box]) / alpha[i][box].size
        assert kept > 0.99 if tracked[i] else kept == 0, (i, kept)
