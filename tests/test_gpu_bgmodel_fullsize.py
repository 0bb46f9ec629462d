"""regionfill and BackgroundAgent.forward on the device at 1080p and 4K.

regionfill is conjugate gradients in float64 (csrc/vu_regionfill.cu) where the reference calls scipy's direct spsolve, so
its contract is a tolerance: <= 1e-5 grey levels on the float result, <= 1 LSB on <= 1e-4 of the filled pixels after the
reference's truncation to uint8, the unmasked pixels untouched.  The cases are the ones where an iterative solve is least
certain: person-sized holes at full size, holes on the image border (masked pixels with 3 or 2 in-image neighbours), many
small components, solutions that are integers (the snap), near-full masks (the largest condition numbers: compared with
closed forms where spsolve is too slow, and with oracle/refport.py:laplace_residual) and odd sizes at factor 0.5.
BackgroundAgent 'mean' and 'pcov' are bit-exact against oracle/refport.py:background_forward at working sizes 540, 960 and
1920, 'pcov' also on holes that finish at chosen round counts around the 8-round read-back and the 100-round cap."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

from scipy.ndimage import distance_transform_cdt  # noqa: E402

from oracle import cvmodel as cvm  # noqa: E402
from oracle import refport as R  # noqa: E402
from test_oracle_laplace import toprow_fill  # noqa: E402
from video_unscreen_b200 import synth  # noqa: E402

HD, UHD = (1080, 1920), (2160, 3840)
TOL = 1e-5          # grey levels, float result
FLIPS = 1e-4        # share of the filled pixels whose truncated uint8 value may differ (by 1)
ON_INT = 1e-9       # a reference value this close to an integer is that integer up to spsolve's own round-off
RESID = 1e-5        # laplace_residual of a device fill (max norm): the snap to integers moves a value by up to 1e-6,
                    # which is up to 8e-6 in the residual; the stop at |r|_2 <= 1e-10 |b|_2 leaves ~1e-7


@pytest.fixture(scope="module")
def U():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import video_unscreen_b200.unscreen.utils as U
    return U


@pytest.fixture(scope="module")
def ops(U):
    from video_unscreen_b200 import ops
    return ops


_cache = {}


def cached(key, fn):
    """oracle results are shared between the tests of this module (spsolve at 4K takes tens of seconds)"""
    if key not in _cache:
        _cache[key] = fn()
    return _cache[key]


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def frame(h, w, seed=0):
    """textured background plus noise, uint8 BGR"""
    rng = np.random.default_rng([seed, h, w])
    img = synth.textured_background(h, w, seed).astype(np.int16) + rng.integers(-8, 9, (h, w, 3))
    return np.clip(img, 0, 255).astype(np.uint8)


def person(h, w):
    """a person-sized ellipse (about 276 k pixels at 1080p)"""
    return synth.ellipse_mask(h, w, 0.5 * w, 0.55 * h, 0.14 * w, 0.3 * h)


def grey_matte(h, w, seed=0):
    """a person matte up-scaled from 1/8 size: grey values 1..254 on its edges, a few grey specks"""
    small = person(h // 8, w // 8).astype(np.uint8) * 255
    m = cvm.resize_linear(small, w, h)
    rng = np.random.default_rng(seed)
    specks = rng.random((h, w)) < 2e-4
    m[specks] = rng.integers(1, 255, int(specks.sum()))
    assert ((m > 0) & (m < 255)).sum() > 1000
    return m


def check_fill(got, want, plane, m):
    """the regionfill contract for one plane; -> max |difference|.  Where the exact fill is an integer, spsolve lands within
    ~1e-12 on either side of it and its own round-off decides the reference's truncated level (a one-pixel boundary: every
    filled pixel one level low; salt at density 0.3: 2.4e-4 of them); there the device must give the integer itself"""
    m = m != 0
    assert got.dtype == np.float64 and got.shape == want.shape
    d = float(np.abs(got - want).max())
    assert d <= TOL, d
    g, r = got[m], want[m]
    on_int = np.abs(r - np.rint(r)) <= ON_INT
    assert np.array_equal(g[on_int], np.rint(r[on_int]))
    gt, rt = g[~on_int].astype(np.int32), r[~on_int].astype(np.int32)
    assert (gt != rt).sum() <= FLIPS * g.size, (gt != rt).sum() / g.size
    assert gt.size == 0 or np.abs(gt - rt).max() <= 1
    assert np.array_equal(got[~m], np.asarray(plane, np.float64)[~m])
    return d


def spsolve(key, plane, m, factor=1.0):
    return cached(("rf", key, factor), lambda: R.regionfill(plane, m, factor))


# ---- regionfill ------------------------------------------------------------------------------------------------


def test_regionfill_person_1080p_three_planes(U):
    """bg.py:79: the B, G, R planes share one mask and are solved together; each equals spsolve and its own solve alone;
    a second run agrees (float64 atomics: not bit-equal); factor 0.5 as the agent calls it"""
    h, w = HD
    planes = np.ascontiguousarray(frame(h, w, 1).transpose(2, 0, 1))
    m = person(h, w)
    m255 = m.astype(np.uint8) * 255
    got3 = U.regionfill(dev(planes), dev(m255), 1.0)
    again = U.regionfill(dev(planes), dev(m255), 1.0)
    assert float((got3 - again).abs().max()) <= TOL
    got3 = got3.cpu().numpy()
    for c in range(3):
        check_fill(got3[c], spsolve(("person_hd", c), planes[c], m), planes[c], m)
        alone = U.regionfill(planes[c], m)
        assert np.abs(alone - got3[c]).max() <= TOL
    assert R.laplace_residual(got3, planes, m) <= RESID
    check_fill(U.regionfill(planes[1], m255, 0.5), spsolve(("person_hd", 1), planes[1], m, 0.5), planes[1], m)


def test_regionfill_person_4k(U):
    """1.27 M unknowns: one plane against spsolve, all three by their residual"""
    h, w = UHD
    planes = np.ascontiguousarray(frame(h, w, 2).transpose(2, 0, 1))
    m = person(h, w)
    got3 = U.regionfill(dev(planes), dev(m), 1.0).cpu().numpy()
    check_fill(got3[0], spsolve("person_4k", planes[0], m), planes[0], m)
    assert R.laplace_residual(got3, planes, m) <= RESID
    for c in (1, 2):
        assert np.array_equal(got3[c][~m], planes[c][~m].astype(np.float64))


def border_holes(h, w):
    """holes along the top, bottom, left and right edges, in the four corners, and one from the top to the bottom edge"""
    m = np.zeros((h, w), bool)
    m[:150, 300:700] = True                     # top edge
    m[h - 120:, 900:1300] = True                # bottom edge
    m[400:700, :180] = True                     # left edge
    m[200:500, w - 90:] = True                  # right edge
    for ys, xs in ((slice(0, 100), slice(0, 140)), (slice(0, 60), slice(w - 200, w)), (slice(h - 130, h), slice(0, 90)),
                   (slice(h - 70, h), slice(w - 110, w))):
        m[ys, xs] = True
    m[:, 1500:1540] = True                      # splits the frame: pixels with only 2 horizontal neighbours in the mask
    return m


@pytest.mark.parametrize("factor", [1.0, 0.5])
def test_regionfill_border_holes(U, factor):
    """masked pixels on the image border have 3 (edges) or 2 (corners) in-image neighbours; the bounding box of the solve
    cannot grow past the image there"""
    h, w = HD
    plane = frame(h, w, 3)[:, :, 2]
    m = border_holes(h, w)
    check_fill(U.regionfill(plane, m, factor), spsolve("border", plane, m, factor), plane, m)


def test_regionfill_salt(U):
    """about 180 k separate components (salt at density 0.3): one solve for all of them"""
    h, w = HD
    plane = frame(h, w, 4)[:, :, 0]
    m = np.random.default_rng(4).random((h, w)) < 0.3
    got = U.regionfill(plane, m)
    check_fill(got, spsolve("salt", plane, m), plane, m)
    assert R.laplace_residual(got, plane, m) <= RESID


def test_regionfill_integer_solutions(U):
    """where the exact fill is an integer, the truncated value must be that integer, not one below it: a checkerboard of
    isolated pixels whose neighbours are multiples of 4 (every interior fill is an integer), and a flat plane"""
    h, w = HD
    yy, xx = np.indices((h, w))
    m = (yy + xx) % 2 == 0
    plane = (np.random.default_rng(5).integers(0, 64, (h, w)) * 4).astype(np.uint8)
    got = U.regionfill(plane, m)
    want = spsolve("checker", plane, m)
    check_fill(got, want, plane, m)
    assert np.array_equal(got.astype(np.uint8), want.astype(np.uint8))
    inner = m.copy()
    inner[[0, -1], :] = inner[:, [0, -1]] = False
    assert np.array_equal(got[inner], np.rint(got[inner]))
    flat = np.full((h, w), 77, np.uint8)
    for factor in (1.0, 0.5):
        assert np.array_equal(U.regionfill(flat, person(h, w), factor), flat.astype(np.float64))


def near_full(h, w, kind):
    m = np.ones((h, w), bool)
    if kind == "toprow":
        m[0] = False
    else:
        m[h // 3, (2 * w) // 3] = False
    return m


def exact_near_full(plane, m, kind):
    """the fill in closed form: the top-row case is separable (toprow_fill); with one boundary pixel the harmonic fill is
    that pixel's value everywhere (the image border adds no boundary data)"""
    if kind == "toprow":
        out = toprow_fill(plane[0], plane.shape[0])
        out[0] = plane[0]
        return out
    return np.full(plane.shape, float(plane[~m][0]))


@pytest.mark.parametrize("kind", ["toprow", "onepixel"])
def test_regionfill_near_full_against_spsolve(U, kind):
    """every pixel but the top row / but one pixel at 540 x 960: the largest condition numbers at a size spsolve solves"""
    h, w = 540, 960
    plane = frame(h, w, 6)[:, :, 1]
    m = near_full(h, w, kind)
    want = spsolve(("near_full", kind), plane, m)
    assert np.abs(want - exact_near_full(plane, m, kind)).max() <= 1e-8
    got = U.regionfill(plane, m)
    check_fill(got, want, plane, m)
    assert R.laplace_residual(got, plane, m) <= RESID


@pytest.mark.parametrize("size", [HD, UHD], ids=["1080p", "4k"])
@pytest.mark.parametrize("kind", ["toprow", "onepixel"])
def test_regionfill_near_full_fullsize(U, ops, kind, size):
    """the near-full masks at 1080p and 4K (2 M and 8.3 M unknowns), against their closed forms: the solve must converge
    (no RuntimeError) and keep the tolerance"""
    h, w = size
    plane = frame(h, w, 7)[:, :, 0]
    m = near_full(h, w, kind)
    out, iters = ops.laplace_fill(dev(plane[None]).double(), dev(m.astype(np.uint8)))
    got = out[0].cpu().numpy()
    check_fill(got, exact_near_full(plane, m, kind), plane, m)
    assert R.laplace_residual(got, plane, m) <= RESID
    print(f"{kind} {h}x{w}: {iters} iterations")


@pytest.mark.parametrize("size", [(1079, 1919), (1081, 1921)], ids=["1079x1919", "1081x1921"])
def test_regionfill_odd_sizes_half(U, ops, size):
    """factor 0.5 on odd sizes: 1079 x 1919 halves to 540 x 960 (rounded half to even) with a last row and column that
    average what exists in float32 (cv2's INTER_AREA tail); 1081 x 1921 halves to 540 x 960 too, dropping the last source
    row and column.  Holes reach the last row and column, so the tail feeds the boundary data and the paste back up"""
    h, w = size
    rng = np.random.default_rng(h)
    plane = frame(h, w, 8)[:, :, 1].astype(np.float64) + rng.random((h, w))      # fractional: float32 rounding shows
    m = person(h, w)
    m[h - 200:, w - 300:] = True
    m[h - 1, 100:400] = True
    check_fill(U.regionfill(plane, m, 0.5), spsolve(("odd", h), plane, m, 0.5), plane, m)
    # the two resizes themselves against the model (no solve in between)
    dh, dw = cvm.scaled_size(h, 0.5), cvm.scaled_size(w, 0.5)
    assert (dh, dw) == (540, 960)
    lo = ops.resize_linear_f64(dev(plane[None]), dh, dw, 0.5, 0.5)
    want_lo = cvm.resize_linear_f64(plane, dw, dh, 0.5, 0.5)
    assert np.abs(lo[0].cpu().numpy() - want_lo).max() <= 1e-9
    up = ops.resize_linear_f64(lo, h, w, keep_mask=dev(m.astype(np.uint8)), keep_src=dev(plane[None]))[0].cpu().numpy()
    want_up = cvm.resize_linear_f64(want_lo, w, h)
    assert np.abs(up[m] - want_up[m]).max() <= 1e-9
    assert np.array_equal(up[~m], plane[~m])


# ---- BackgroundAgent -------------------------------------------------------------------------------------------


def agent_case(size, seed):
    h, w = size
    return frame(h, w, seed), grey_matte(h, w, seed)


def check_agent(img, m, L, key, methods=("mean", "pcov", "rf"), **kw):
    from video_unscreen_b200.unscreen.bgmodel import BackgroundAgent
    ag = BackgroundAgent(input_long_side=L, **kw)
    for method in methods:
        got = ag.forward(img, m, method)
        want = cached(("agent", key, L, method, tuple(sorted(kw.items()))),
                      lambda: R.background_forward(img, m, method, input_long_side=L, **kw))
        assert got.dtype == want.dtype and got.shape == want.shape
        if method == "rf":
            diff = np.abs(got.astype(np.int32) - want.astype(np.int32))
            assert diff.max() <= 1 and (diff > 0).mean() <= 1e-3, (L, diff.max(), (diff > 0).mean())
        else:
            assert np.array_equal(got, want), (L, method, int((got != want).sum()))


ALL = ("mean", "pcov", "rf")


@pytest.mark.parametrize("size,L,methods", [(HD, 540, ALL), (HD, 960, ALL), (HD, 1920, ("mean", "rf")), (UHD, 540, ALL),
                                            (UHD, 1920, ALL)],
                         ids=["1080p-540", "1080p-960", "1080p-1920", "4k-540", "4k-1920"])
def test_agent_forward(U, size, L, methods):
    """'mean' / 'pcov' bit-exact, 'rf' <= 1 LSB on <= 1e-3 of the values, on a grey matte; at 960 and more the hole is
    wider than 400 px at the working size, so 'pcov' stops at its 100-round cap (the oracle's 100 rounds on a 1920 x 1080
    working image take most of a minute: once, from the 4K frame)"""
    img, m = agent_case(size, 11)
    check_agent(img, m, L, size, methods)


@pytest.mark.parametrize("k,dk,di", [(3, 3, 2), (7, 7, 3)])
def test_agent_pcov_ksize(U, k, dk, di):
    img, m = agent_case(HD, 12)
    check_agent(img, m, 960, "ksize", ("pcov",), pcov_ksize=k, dilation_ksize=dk, dilation_iters=di)


@pytest.mark.parametrize("rounds", [1, 7, 8, 9, 16, 17, 99, 100, 101])
def test_pcov_round_counts(U, ops, rounds):
    """square holes that 'pcov' (k = 5) fills in exactly 1 ... 101 rounds: a hole pixel at chessboard distance d from a valid
    pixel turns valid in round ceil(d / 2).  101 rounds is past the cap: the centre stays invalid (0).  Reading the flags
    back after every round, every 8 rounds or once gives the same box, and the oracle's"""
    k, s = 5, 4 * rounds
    h, w = max(2 * s, 64), max(2 * s, 64) + 37
    img = frame(h, w, rounds)
    m = np.zeros((h, w), np.uint8)
    y0, x0 = (h - s) // 2, (w - s) // 2
    m[y0:y0 + s, x0:x0 + s] = 200
    d = distance_transform_cdt(m > 0, metric="chessboard")
    assert int(np.ceil(d.max() / (k // 2))) == rounds
    box = tuple(int(v) for v in R.get_fgbox(m, padsize=k))
    want = R.bg_by_pcov(img, m, k)[box[0]:box[1], box[2]:box[3]]
    outs = [ops.pcov_fill(dev(img), dev(m), box, k, batch=b).cpu().numpy() for b in (1, 8, 100)]
    for got in outs:
        assert np.array_equal(got, want)
    c = (h // 2 - box[0], w // 2 - box[2])
    assert not want[c].any() if rounds > 100 else want[c].any()


@pytest.mark.parametrize("where", ["corner", "edge"])
def test_pcov_box_on_the_border(U, ops, where):
    """the box around the hole is clamped by the image: the box filter reflects at the box edge, which is the image edge
    on the clamped sides"""
    h, w = HD
    img = frame(h, w, 13)
    m = np.zeros((h, w), np.uint8)
    if where == "corner":
        m[:90, w - 140:] = 255
    else:
        m[300:520, :60] = 255
    box = tuple(int(v) for v in R.get_fgbox(m, padsize=5))
    got = ops.pcov_fill(dev(img), dev(m), box, 5).cpu().numpy()
    assert np.array_equal(got, R.bg_by_pcov(img, m, 5)[box[0]:box[1], box[2]:box[3]])
    mm = np.zeros((h, w), np.uint8)
    if where == "corner":
        mm[:200, w - 300:] = 255
    else:
        mm[400:900, :120] = 255
    check_agent(img, mm, 960, ("border", where), ("pcov", "mean"))


def test_empty_boundary(U, ops):
    """a mask that is 255 but for one pixel escapes the all-foreground early-out, but after the resize and the dilation
    the working mask is everywhere and its outer boundary empty: 'mean' takes the whole image's mean colour, 'pcov' runs
    its 100 rounds with nothing valid, both bit-exact.  'rf' has no boundary data at all, the Laplace system is singular
    (spsolve returns NaN); the device's solve starts from 0 with a zero right-hand side and returns 0 at once: V = 0, so
    the background is black"""
    from video_unscreen_b200.unscreen.bgmodel import BackgroundAgent
    h, w = HD
    img = frame(h, w, 14)
    m = np.full((h, w), 255, np.uint8)
    m[500, 700] = 0
    for L in (540, 960):
        check_agent(img, m, L, "full", ("mean", "pcov"))
        got = BackgroundAgent(input_long_side=L).forward(img, m, "rf")
        assert got.dtype == np.uint8 and got.shape == img.shape and not got.any()
    out, iters = ops.laplace_fill(torch.full((2, 30, 40), 9.0, dtype=torch.float64, device="cuda"),
                                  torch.ones((30, 40), dtype=torch.uint8, device="cuda"))
    assert iters == 0 and not out.any()


def test_mask_bbox_and_masked_sum3_4k(U, ops):
    h, w = UHD
    img = frame(h, w, 15)
    m = grey_matte(h, w, 15)
    ys, xs = np.nonzero(m)
    assert ops.mask_bbox(dev(m)) == (ys.min(), ys.max(), xs.min(), xs.max())
    one = np.zeros((h, w), np.uint8)
    one[h - 1, w - 1] = 1
    assert ops.mask_bbox(dev(one)) == (h - 1, h - 1, w - 1, w - 1)
    assert ops.mask_bbox(dev(np.zeros_like(one))) is None
    sums, n = ops.masked_sum3(dev(img), dev(m))
    assert n == len(ys) and sums == img[m > 0].astype(np.int64).sum(axis=0).tolist()
    sums, n = ops.masked_sum3(dev(img))
    assert n == h * w and sums == img.reshape(-1, 3).astype(np.int64).sum(axis=0).tolist()
