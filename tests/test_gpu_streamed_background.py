"""Streamed temporal backgrounds: the median and masked-mean accumulators (vu_median_accum_*, vu_masked_mean_accum_*),
their ops classes and the clip.streamed_* helpers.  A clip added in any chunking and any chunk order must give the bytes
of the resident-clip call: np.median(stack, 0).astype(uint8) for the median, bg_offline.py:106-125 for the mean.  The
argument checks of the C ABI run without a GPU; everything else is marked ``gpu``."""
import ctypes

import numpy as np
import pytest

from oracle import refport as R
from video_unscreen_b200 import _lib, synth

torch = pytest.importorskip("torch")

gpu = pytest.mark.gpu


# ---- C ABI argument checks: no kernel is launched -----------------------------------------------------------------------

def test_accumulator_abi_refuses_bad_arguments_without_a_gpu():
    L = _lib.lib()
    null = ctypes.c_void_p(0)
    st = ctypes.c_void_p(1 << 20)     # never dereferenced: every call below is refused before it touches memory
    fr = ctypes.c_void_p(2 << 20)
    inval = -1
    assert L.vu_median_accum_bytes(1) == L.vu_median_accum_bytes(128) == 128 * 512
    assert L.vu_median_accum_bytes(129) == 256 * 512
    assert L.vu_median_accum_bytes(0) == 0
    assert L.vu_masked_mean_accum_bytes(3, 5) == 3 * 5 * 16
    # null pointers
    assert L.vu_median_accum_reset(null, 64, null) == inval
    assert L.vu_median_accum_add_u8(null, 64, fr, 1, 0, null) == inval
    assert L.vu_median_accum_add_u8(st, 64, null, 1, 0, null) == inval
    assert L.vu_median_accum_finish_u8(null, 64, 1, fr, null) == inval
    assert L.vu_median_accum_finish_u8(st, 64, 1, null, null) == inval
    # k < 1
    assert L.vu_median_accum_add_u8(st, 64, fr, 0, 0, null) == inval
    assert L.vu_median_accum_add_u8(st, 64, fr, -3, 10, null) == inval
    # n_before + k > 65535 (16-bit counters)
    assert L.vu_median_accum_add_u8(st, 64, fr, 1, 65535, null) == inval
    assert L.vu_median_accum_add_u8(st, 64, fr, 65536, 0, null) == inval
    assert L.vu_median_accum_add_u8(st, 64, fr, 2, 65534, null) == inval
    assert L.vu_median_accum_add_u8(st, 64, fr, 1, -1, null) == inval
    # finish with n < 1 (or beyond the counters)
    assert L.vu_median_accum_finish_u8(st, 64, 0, fr, null) == inval
    assert L.vu_median_accum_finish_u8(st, 64, 65536, fr, null) == inval
    # a state that is not 16-byte aligned
    assert L.vu_median_accum_add_u8(ctypes.c_void_p((1 << 20) + 4), 64, fr, 1, 0, null) == inval
    # masked mean
    assert L.vu_masked_mean_accum_reset(null, 4, 4, null) == inval
    assert L.vu_masked_mean_accum_add(null, fr, fr, 1, 16, null) == inval
    assert L.vu_masked_mean_accum_add(st, null, fr, 1, 16, null) == inval
    assert L.vu_masked_mean_accum_add(st, fr, null, 1, 16, null) == inval
    assert L.vu_masked_mean_accum_add(st, fr, fr, 0, 16, null) == inval
    assert L.vu_masked_mean_accum_add_dilate32(null, fr, fr, 1, 4, 16, null) == inval
    assert L.vu_masked_mean_accum_add_dilate32(st, fr, null, 1, 4, 16, null) == inval
    assert L.vu_masked_mean_accum_add_dilate32(st, fr, fr, 0, 4, 16, null) == inval
    assert L.vu_masked_mean_accum_finish(null, 16, 10, fr, fr, null) == inval
    assert L.vu_masked_mean_accum_finish(st, 16, 10, null, fr, null) == inval


# ---- helpers --------------------------------------------------------------------------------------------------------------

def _need_cuda():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")


def _cuda(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _spans(n, sizes=(1, 7, 64)):
    """[s, e) chunks of the given sizes, then the remainder"""
    out, s = [], 0
    for z in sizes:
        if s >= n:
            break
        out.append((s, min(n, s + z)))
        s = out[-1][1]
    if s < n:
        out.append((s, n))
    return out


def _permuted(n, seed):
    spans = _spans(n, (1, 7, 64, 5, 33))
    order = np.random.default_rng(seed).permutation(len(spans))
    return [spans[i] for i in order]


def _column_clip(n, h, w):
    """the column-dependent pattern of test_gpu_median_columns: every byte has its own median"""
    m = h * w * 3
    e = np.arange(m)
    mu = ((e % 16) * 16 + (e // 16) % 16).astype(np.int16)
    rng = np.random.default_rng(n)
    return np.clip(mu[None] + rng.integers(-3, 4, (n, m)), 0, 255).astype(np.uint8).reshape(n, h, w, 3)


def _clip(kind, n, h=16, w=50):
    if kind == "columns":
        return _column_clip(n, h, w)
    if kind == "random":
        return synth.random_clip(n, h, w, seed=n)
    return synth.bgstep_clip(n, h, w, seed=n)[0]


def _median_four_ways(frames):
    """the accumulator's result for the clip added in one chunk, in uneven chunks, in permuted chunks and after a reset
    that followed a different clip"""
    from video_unscreen_b200 import ops
    d = _cuda(frames)
    n = d.shape[0]
    acc = ops.TemporalMedianAccumulator(d.shape[1:])
    got = {}
    acc.add(d)
    got["one chunk"] = acc.result().cpu().numpy()
    acc.reset()
    for s, e in _spans(n):
        acc.add(d[s:e])
    got["uneven chunks"] = acc.result().cpu().numpy()
    acc.reset()
    for s, e in _permuted(n, n):
        acc.add(d[s:e])
    got["permuted chunks"] = acc.result().cpu().numpy()
    acc.reset()
    acc.add(_cuda(synth.random_clip(37, *frames.shape[1:3], seed=5)))
    acc.reset()
    for s, e in _spans(n, (3, 50)):
        acc.add(d[s:e])
    got["after reset"] = acc.result().cpu().numpy()
    assert acc.n == n
    return got


def _assert_same(got, want, what):
    bad = np.flatnonzero(got.reshape(-1) != want.reshape(-1))
    assert bad.size == 0, f"{what}: {bad.size} bytes differ, first at {bad[:8].tolist()}"


# ---- median ----------------------------------------------------------------------------------------------------------------

@gpu
@pytest.mark.parametrize("kind", ["columns", "random", "bgstep"])
@pytest.mark.parametrize("n", [1, 2, 3, 299, 300, 1000])
def test_median_accumulator_matches_oracle(n, kind):
    _need_cuda()
    frames = _clip(kind, n)
    want = R.temporal_median(frames)
    for way, got in _median_four_ways(frames).items():
        _assert_same(got, want, way)


@pytest.fixture(scope="module")
def bgstep_1080p():
    frames, masks, _ = synth.bgstep_clip(300, 1080, 1920, seed=3)
    return frames, masks


@gpu
def test_median_accumulator_matches_resident_kernel_1080p(bgstep_1080p):
    _need_cuda()
    from video_unscreen_b200 import ops
    d = _cuda(bgstep_1080p[0])
    want = ops.temporal_median(d)
    acc = ops.TemporalMedianAccumulator(d.shape[1:])
    for s, e in _spans(300, (1, 7, 64, 100)):
        acc.add(d[s:e])
    assert torch.equal(acc.result(), want)


@gpu
def test_median_accumulator_matches_two_pass_kernel_n1000():
    _need_cuda()
    from video_unscreen_b200 import ops
    d = _cuda(synth.bgstep_clip(1000, 72, 128, seed=11)[0])
    want = ops.temporal_median(d)     # > 608 frames with a workspace: estimate + refine + fix-up
    acc = ops.TemporalMedianAccumulator(d.shape[1:])
    for s, e in _permuted(1000, 3):
        acc.add(d[s:e])
    assert torch.equal(acc.result(), want)


@gpu
@pytest.mark.parametrize("shape", [(7, 13, 3), (10, 30, 3), (5, 41), (1,)])
def test_median_accumulator_odd_shapes_and_unaligned_frames(shape):
    """m not a multiple of 16 (or of 4), a last tile that is partly outside the frame, and frames whose base address is
    one byte off 16-byte alignment"""
    _need_cuda()
    from video_unscreen_b200 import ops
    n = 75
    m = int(np.prod(shape))
    frames = np.random.default_rng(m).integers(0, 256, (n,) + shape, dtype=np.uint8)
    want = R.temporal_median(frames)
    buf = torch.empty(n * m + 1, dtype=torch.uint8, device="cuda")
    off = buf[1:].view((n,) + shape)
    off.copy_(_cuda(frames))
    assert off.data_ptr() % 16 == 1
    d = _cuda(frames)
    for src, what in ((d, "aligned"), (off, "one byte off")):
        acc = ops.TemporalMedianAccumulator(shape)
        for s, e in _spans(n, (2, 9, 30)):
            acc.add(src[s:e])
        _assert_same(acc.result().cpu().numpy(), want, what)


@gpu
def test_median_accumulator_counter_limit():
    _need_cuda()
    from video_unscreen_b200 import ops
    # 300 bytes: two whole 128-byte tiles (vector loads) and a partial one (byte loads)
    frames = torch.full((65535, 300), 200, dtype=torch.uint8, device="cuda")
    frames[:, 1::2] = 7                 # the two counters of a word in different bins
    frames[:, 32:64] = 255              # ... and in the same bin
    frames[:, 260:] = 255
    acc = ops.TemporalMedianAccumulator((300,))
    for s, e in _spans(65535, (1, 8191, 30000)):
        acc.add(frames[s:e])
    assert acc.n == 65535
    want = frames[0].clone()
    assert torch.equal(acc.result(), want)
    before = acc.state.clone()
    with pytest.raises(_lib.VuError):
        acc.add(frames[:1])
    assert acc.n == 65535
    torch.cuda.synchronize()
    assert torch.equal(acc.state, before)
    assert torch.equal(acc.result(), want)


# ---- masked mean -----------------------------------------------------------------------------------------------------------

def _mean_clip(n, h, w, seed):
    """random frames; sparse masked pixels of the values that matter (255 drops the frame, >= 250 stops the count, 249
    and 100 do neither), and a block that is never unmasked"""
    rng = np.random.default_rng(seed)
    frames = rng.integers(0, 256, (n, h, w, 3), dtype=np.uint8)
    masks = np.zeros((n, h, w), np.uint8)
    sel = rng.random((n, h, w)) < 0.04
    masks[sel] = rng.choice(np.array([100, 249, 250, 254, 255], np.uint8), size=int(sel.sum()))
    masks[:, :5, :7] = 255
    return frames, masks


def _counts(masks, ksize, iters):
    return sum((R.dilate_mask(m, ksize, iters) < 250).astype(np.int64) for m in masks)


@gpu
@pytest.mark.parametrize("h,w,ksize,iters", [(40, 64, 3, 2), (40, 50, 3, 2), (40, 64, 5, 1), (37, 51, 3, 1)])
def test_masked_mean_accumulator(h, w, ksize, iters):
    """fused (3, 2) path (w % 16 == 0), the generic path (w % 16 != 0, other structuring elements, h * w not a multiple
    of 4); min_count is picked so that pixels with exactly min_count and min_count + 1 counted frames exist"""
    _need_cuda()
    from video_unscreen_b200 import ops
    n = 40
    frames, masks = _mean_clip(n, h, w, seed=h * w + ksize)
    cnt = _counts(masks, ksize, iters)
    min_count = int(np.median(cnt))
    assert (cnt == min_count).any() and (cnt == min_count + 1).any() and (cnt == 0).any()
    want_bg, want_always = R.masked_temporal_mean(frames, masks, ksize, iters, min_count)
    fd, md = _cuda(frames), _cuda(masks)
    resident = None
    if (h * w) % 4 == 0:
        resident = [t.cpu().numpy() for t in ops.masked_temporal_mean_raw(fd, md, ksize, iters, min_count)]
        assert np.array_equal(resident[0], want_bg) and np.array_equal(resident[1], want_always)
    acc = ops.MaskedMeanAccumulator(h, w, ksize, iters, min_count)
    fused = (ksize, iters) == (3, 2) and w % 16 == 0
    for spans in (_spans(n, (1, 7, 13)), _permuted(n, 1), [(0, n)]):
        acc.reset()
        for s, e in spans:
            before = _lib.lib().vu_launch_count()
            acc.add(fd[s:e], md[s:e])
            if fused:
                assert _lib.lib().vu_launch_count() - before == 1, "the fused add should be one launch"
        bg, always = (t.cpu().numpy() for t in acc.result())
        _assert_same(bg, want_bg, f"bg, chunks {spans}")
        _assert_same(always, want_always, f"mask_always, chunks {spans}")
    assert acc.n == n


# ---- streamed helpers --------------------------------------------------------------------------------------------------------

def _batches(d, size):
    """device batches as parallel_read_img(..., on_device=True) returns them: lists of [H, W, 3] tensors"""
    for s in range(0, d.shape[0], size):
        yield [d[i] for i in range(s, min(d.shape[0], s + size))]


@gpu
def test_streamed_temporal_median(bgstep_1080p):
    _need_cuda()
    from video_unscreen_b200 import clip, ops
    frames = bgstep_1080p[0]
    d = _cuda(frames)
    want = ops.temporal_median(d)
    pinned = torch.from_numpy(frames).pin_memory()
    assert torch.equal(clip.streamed_temporal_median(pinned, chunk=64), want)
    assert torch.equal(clip.streamed_temporal_median(frames, chunk=100, depth=3), want)
    assert torch.equal(clip.streamed_temporal_median(_batches(d, 64)), want)
    assert torch.equal(clip.streamed_temporal_median(d[s:e] for s, e in _spans(300)), want)


@gpu
@pytest.mark.parametrize("h,w", [(128, 192), (96, 200)])
def test_streamed_masked_temporal_mean(h, w):
    _need_cuda()
    from video_unscreen_b200 import clip, ops
    frames, masks, _ = synth.bgstep_clip(120, h, w, seed=4)
    fd, md = _cuda(frames), _cuda(masks)
    want = [t.cpu().numpy() for t in ops.masked_temporal_mean_raw(fd, md)]
    runs = {
        "pinned": clip.streamed_masked_temporal_mean(torch.from_numpy(frames).pin_memory(), torch.from_numpy(masks).pin_memory(), chunk=50),
        "numpy": clip.streamed_masked_temporal_mean(frames, masks, chunk=33),
        "device batches": clip.streamed_masked_temporal_mean(_batches(fd, 64), (md[s:s + 64] for s in range(0, 120, 64))),
    }
    for what, (bg, always) in runs.items():
        _assert_same(bg.cpu().numpy(), want[0], what)
        _assert_same(always.cpu().numpy(), want[1], what)


# ---- streams and graphs ------------------------------------------------------------------------------------------------------

@gpu
def test_accumulators_on_a_side_stream_and_in_a_graph():
    _need_cuda()
    from video_unscreen_b200 import clip, ops
    a = synth.bgstep_clip(50, 48, 64, seed=8)
    b = synth.bgstep_clip(50, 48, 64, seed=9)
    frames = np.concatenate([a[0], b[0]])
    masks = np.concatenate([a[1], b[1]])
    want_med = R.temporal_median(frames)
    want_mean = R.masked_temporal_mean(frames, masks)

    # side stream
    acc = ops.TemporalMedianAccumulator(frames.shape[1:])
    macc = ops.MaskedMeanAccumulator(48, 64)
    fd, md = _cuda(frames), _cuda(masks)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        acc.add(fd[:50]).add(fd[50:])
        macc.add(fd[:50], md[:50]).add(fd[50:], md[50:])
    torch.cuda.current_stream().wait_stream(side)
    _assert_same(acc.result().cpu().numpy(), want_med, "median, side stream")
    bg, always = macc.result()
    _assert_same(bg.cpu().numpy(), want_mean[0], "mean, side stream")
    _assert_same(always.cpu().numpy(), want_mean[1], "mask_always, side stream")

    # captured add: the warm-up run adds the first half, the replay the second half refilled into the same buffers
    acc.reset()
    macc.reset()
    fbuf, mbuf = fd[:50].clone(), md[:50].clone()
    g = clip.Graphed(lambda: (acc.add(fbuf), macc.add(fbuf, mbuf)))
    assert acc.n == 100 and macc.n == 100      # counted at the warm-up and at the capture
    fbuf.copy_(fd[50:])
    mbuf.copy_(md[50:])
    g.replay()
    _assert_same(acc.result().cpu().numpy(), want_med, "median, graph replay")
    bg, always = macc.result()
    _assert_same(bg.cpu().numpy(), want_mean[0], "mean, graph replay")
    _assert_same(always.cpu().numpy(), want_mean[1], "mask_always, graph replay")

    # an add captured while the accumulator is empty (.n == 0) still accumulates on every replay
    acc2 = ops.TemporalMedianAccumulator(frames.shape[1:])
    fbuf.copy_(fd[:50])
    acc2.add(fbuf).reset()              # a first launch outside the capture, then empty again
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        acc2.add(fbuf)
    assert acc2.n == 50
    graph.replay()
    fbuf.copy_(fd[50:])
    graph.replay()
    acc2.n = 100                        # two replays of 50 frames, counted by the caller
    _assert_same(acc2.result().cpu().numpy(), want_med, "median, graph captured with n == 0")
