"""Batched, device-resident clip pipelines: the per-frame stages of the
reference's pipeline scripts run over [N,H,W,...] stacks with no host round
trip (per-frame branches are taken on the device), which is how the per-frame
hot path gets anywhere near the HBM roofline (a 1080p stage moves ~10 MB: less
than one kernel launch).  Results are identical, frame by frame, to the
per-frame agents in ``video_unscreen_b200.unscreen`` (tests/test_gpu_clip.py).

Frames are processed in chunks so that the low-resolution intermediates stay
L2-resident between the kernels that produce and consume them.
"""
import numpy as np
import torch

from . import _lib, ops
from .unscreen.utils.fgfuncs import bgr2hsv_pixel
from .unscreen.utils.imgprocess import get_target_size


class Graphed:
    """A clip pipeline captured as ONE CUDA graph: ``Graphed(fn)`` runs ``fn()`` once eagerly (warm-up: kernel
    attributes, allocator), captures a second run, and every ``replay()`` relaunches the whole launch sequence
    (about a hundred kernels for a 300-frame clip) with a single driver call.  The captured kernels read and write
    the very tensors ``fn`` closed over: refill those in place between replays.  ``result`` is what ``fn`` returned
    during capture (tensors owned by the graph's memory pool, overwritten by every replay)."""

    def __init__(self, fn):
        fn()
        torch.cuda.synchronize()
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.result = fn()

    def replay(self):
        self.graph.replay()
        return self.result


def _chunks(n, chunk):
    for s in range(0, n, chunk):
        yield s, min(n, s + chunk)


_SIDE_STREAMS = {}


def _overlap_chunks(n, chunk, body, streams=2):
    """``body(s, e)`` for every chunk [s, e) of n frames.  The chunks of these pipelines are independent, so with
    ``streams`` > 1 consecutive chunks go to alternating side streams: the partial last waves and launch gaps of one
    chunk's kernels are filled by the next chunk's.  Inputs must be ready on the current stream; everything the bodies
    wrote is ready on it at return.  Sequential while a CUDA graph is being captured."""
    spans = list(_chunks(n, chunk))
    if streams <= 1 or len(spans) <= 1 or torch.cuda.is_current_stream_capturing():
        for s, e in spans:
            body(s, e)
        return
    cur = torch.cuda.current_stream()
    key = (cur.device, streams)
    if key not in _SIDE_STREAMS:
        _SIDE_STREAMS[key] = [torch.cuda.Stream(device=cur.device) for _ in range(streams)]
    pool = _SIDE_STREAMS[key][:min(streams, len(spans))]
    ready = torch.cuda.Event()
    ready.record(cur)
    for st in pool:
        st.wait_event(ready)
    for i, (s, e) in enumerate(spans):
        with torch.cuda.stream(pool[i % len(pool)]):
            body(s, e)
    for st in pool:
        done = torch.cuda.Event()
        done.record(st)
        cur.wait_event(done)


_PIPE_STREAMS = {}


def streamed(host_inputs, host_outputs, body, chunk, depth=2):
    """A clip that lives in (pinned) HOST memory through a per-frame clip pipeline, chunk by chunk, with the host->device
    copies, the kernels and the device->host copies of consecutive chunks overlapping on three streams (PCIe is full
    duplex: the step costs max(H2D, D2H), not their sum, and the kernels hide under the copies).

    ``host_inputs`` / ``host_outputs``: lists of CPU tensors [N, ...] (pinned, or the copies are synchronous);
    ``body(s, e, *device_input_chunks, outs)`` runs frames [s, e): ``outs`` are device staging tensors [e - s, ...], one
    per host output, which the body must fill (pass them as ``out=`` to the clip functions).  Chunks must be independent
    (every per-frame stage is).  Returns after the last device->host copy has landed."""
    n = host_inputs[0].shape[0]
    cur = torch.cuda.current_stream()
    dev = cur.device
    if dev not in _PIPE_STREAMS:
        _PIPE_STREAMS[dev] = tuple(torch.cuda.Stream(device=dev) for _ in range(3))
    s_in, s_run, s_out = _PIPE_STREAMS[dev]
    depth = max(1, min(depth, -(-n // chunk)))
    bufs_in = [[torch.empty((chunk,) + tuple(t.shape[1:]), dtype=t.dtype, device=dev) for t in host_inputs] for _ in range(depth)]
    bufs_out = [[torch.empty((chunk,) + tuple(t.shape[1:]), dtype=t.dtype, device=dev) for t in host_outputs] for _ in range(depth)]
    start = torch.cuda.Event()
    start.record(cur)
    for st in (s_in, s_run, s_out):
        st.wait_event(start)
    ran = [None] * depth        # kernels of the chunk that used slot k are done: its input buffers are free
    landed = [None] * depth     # its outputs are on the host: its output buffers are free
    for i, (s, e) in enumerate(_chunks(n, chunk)):
        k = i % depth
        with torch.cuda.stream(s_in):
            if ran[k] is not None:
                s_in.wait_event(ran[k])
            ins = [b[:e - s] for b in bufs_in[k]]
            for b, t in zip(ins, host_inputs):
                b.copy_(t[s:e], non_blocking=True)
            up = torch.cuda.Event()
            up.record(s_in)
        with torch.cuda.stream(s_run):
            s_run.wait_event(up)
            if landed[k] is not None:
                s_run.wait_event(landed[k])
            outs = [b[:e - s] for b in bufs_out[k]]
            body(s, e, *ins, outs)
            ran[k] = torch.cuda.Event()
            ran[k].record(s_run)
        with torch.cuda.stream(s_out):
            s_out.wait_event(ran[k])
            for b, t in zip(outs, host_outputs):
                t[s:e].copy_(b, non_blocking=True)
            landed[k] = torch.cuda.Event()
            landed[k].record(s_out)
    for st in (s_in, s_run, s_out):
        st.synchronize()


def _is_clip(x):
    return isinstance(x, (np.ndarray, torch.Tensor))


def _as_tensor(x):
    return torch.from_numpy(np.ascontiguousarray(x)) if isinstance(x, np.ndarray) else x


def _device_batch(b, dev):
    """one batch [k, ...] of an iterable: a tensor or array, or a list of frames (what parallel_read_img returns)"""
    if isinstance(b, (list, tuple)):
        b = torch.stack([_as_tensor(x) for x in b])
    b = _as_tensor(b)
    return b if b.is_cuda else b.to(dev)


def streamed_temporal_median(host_frames, chunk=256, depth=2, out=None):
    """The exact temporal median (``ops.temporal_median``, byte for byte) of a clip that never has to be on the device in
    one piece.  ``host_frames``: a clip [N, ...] in host memory (a pinned CPU tensor: the host->device copies of chunk i + 1
    overlap the histogram add of chunk i; a numpy array or pageable tensor works too, with synchronous copies), or an
    iterable of batches [k, ...] on the device (e.g. successive ``parallel_read_img(paths, on_device=True)`` results: the
    clip then exists nowhere in full).  Device memory: the accumulator's 512 bytes per frame byte plus ``depth`` chunks.
    At most 65535 frames.  Returns the median as a CUDA tensor of the frame's shape."""
    dev = torch.device("cuda", torch.cuda.current_device())
    if _is_clip(host_frames):
        t = _as_tensor(host_frames)
        acc = ops.TemporalMedianAccumulator(t.shape[1:], dev)
        streamed([t], [], lambda s, e, fr, outs: acc.add(fr), chunk, depth)
    else:
        acc = None
        for b in host_frames:
            b = _device_batch(b, dev)
            if acc is None:
                acc = ops.TemporalMedianAccumulator(b.shape[1:], dev)
            acc.add(b)
        if acc is None:
            raise ValueError("streamed_temporal_median: no frames")
    return acc.result(out)


def streamed_masked_temporal_mean(host_frames, host_masks, chunk=256, ksize=3, iters=2, min_count=10, depth=2):
    """bg_offline.py:106-125 (``ops.masked_temporal_mean_raw``, byte for byte) for a clip fed chunk by chunk:
    ``host_frames`` [N,H,W,3] / ``host_masks`` [N,H,W] (raw masks) in host memory, copied to the device in chunks that
    overlap the accumulation as in ``streamed_temporal_median``, or two iterables of device batches consumed in step.
    Returns (bg [H,W,3], mask_always [H,W]) as CUDA tensors."""
    dev = torch.device("cuda", torch.cuda.current_device())
    if _is_clip(host_frames):
        f, mk = _as_tensor(host_frames), _as_tensor(host_masks)
        acc = ops.MaskedMeanAccumulator(f.shape[1], f.shape[2], ksize, iters, min_count, dev)
        streamed([f, mk], [], lambda s, e, fr, ms, outs: acc.add(fr, ms), chunk, depth)
    else:
        acc = None
        for fb, mb in zip(host_frames, host_masks, strict=True):
            fb, mb = _device_batch(fb, dev), _device_batch(mb, dev)
            if acc is None:
                acc = ops.MaskedMeanAccumulator(fb.shape[1], fb.shape[2], ksize, iters, min_count, dev)
            acc.add(fb, mb)
        if acc is None:
            raise ValueError("streamed_masked_temporal_mean: no frames")
    return acc.result()


def cf_predict_clip(frames, segmasks, agent, chunk=64, out=None, streams=2, return_flags=False):
    """ColorFilteringAgent.forward(frame, mask, iters=0) for every frame of
    frames[N,H,W,3] / segmasks[N,H,W] with the agent's current mixtures
    (reference colorfiltering/agent.py:285-354, predict-only branch :319-321).
    Returns alpha[N,H,W]; the constant background image is ``agent.bg_color_bgr()``.
    ``return_flags``: also the per-frame early-out flags [N] uint8 (1: no foreground, 2: no background: alpha is the
    mask itself, agent.py:303-307; 0: evaluated)."""
    n, h, w, _ = frames.shape
    th, tw = get_target_size(h, w, agent.input_long_side)
    luts = agent.tables_dev()
    lut3d = agent.lut3d_dev()
    alpha = out if out is not None else torch.empty((n, h, w), dtype=torch.uint8, device=frames.device)
    fg_min, bg_min = max(agent.fg_ncomp) * 5, max(agent.bg_ncomp) * 5
    all_flags = torch.empty(n, dtype=torch.uint8, device=frames.device) if return_flags else None

    def body(s, e):
        fr, sm = frames[s:e], segmasks[s:e]
        if ops.cf_lowres_supported(h, w, th, tw):
            # one pass over the frames (the early-out counts of the masks ride along where the pass sees every mask
            # byte), then threshold + d2e2e2d2 marching in registers, then the up-scale
            if ops.cf_lowres_counts_supported(fr, sm, th, tw):
                a_lo, stats, mc = ops.cf_lowres(fr, sm, th, tw, lut3d, want_mask_counts=True)
                flags = ops.degenerate_flags_from_counts(mc, fg_min, bg_min)
            else:
                flags = ops.cf_degenerate_flags(sm, fg_min, bg_min)
                a_lo, stats = ops.cf_lowres(fr, sm, th, tw, lut3d)
            a_lo = ops.cross_chain(a_lo, [(_lib.DILATE, 2), (_lib.ERODE, 2), (_lib.ERODE, 2), (_lib.DILATE, 2)], stats, 0.8)
        else:
            flags = ops.cf_degenerate_flags(sm, fg_min, bg_min)
            hsv_lo = ops.resize_linear_image(ops.bgr2hsv(fr), th, tw)
            a_lo = ops.cf_postprocess(ops.cf_alpha_lut3d(hsv_lo, lut3d), ops.resize_linear_mask(sm, th, tw), 0.8)
        # degenerate masks are returned as they came (agent.py:303-307): alt_src / alt_flags
        ops.resize_up(a_lo, h, w, alt_src=sm, alt_flags=flags, out=alpha[s:e])
        if return_flags:
            all_flags[s:e].copy_(flags)
    _overlap_chunks(n, chunk, body, streams)
    return (alpha, all_flags) if return_flags else alpha


def _trimap_tail(masks, agent, fuzzy=None, flags=None, out=None, work_size=None):
    """nearest down (+ ensemble clearing) -> dilate/erode/classify -> bilinear up + snap (+ fuzzy override); written into
    ``out`` when given.  ``work_size`` overrides the working resolution (row tiles of a frame: the WHOLE frame decides it)."""
    n, h, w = masks.shape
    ih, iw = work_size if work_size is not None else get_target_size(h, w, agent.input_long_side)
    if agent.kernelsize == 3 and ops.trimap_bits_supported(masks, ih, iw, agent.iters, fuzzy):
        # exact 2x / 4x working resolution (1080p, 4K): the whole tail in bit logic, two launches
        return ops.trimap_bits(masks, ih, iw, agent.iters, fuzzy, flags, out=out)
    m = ops.trimap_src_lo(masks, ih, iw, fuzzy, flags)
    if agent.kernelsize == 3 and agent.iters <= ops.CROSS_MAX_PASSES:
        tri = ops.trimap_core(m, agent.iters)
    else:
        tri = ops.trimap_classify(ops.dilate(m, agent.kernelsize, agent.iters), ops.erode(m, agent.kernelsize, agent.iters))
    if (ih, iw) == (h, w) or (ih == 2 * h and iw == 2 * w):   # copy / cv2's INTER_AREA corner cases: unfused tail
        t = ops.trimap_snap(ops.resize_linear_mask(tri, h, w))
        t = ops.set128_unflagged(t, fuzzy, flags) if fuzzy is not None else t
        if out is not None:
            out.copy_(t)
            return out
        return t
    return ops.resize_up(tri, h, w, mode=1, fuzzy=fuzzy, flags=flags, out=out)


def trimap_clip(masks, agent, frames=None, bg=None, chunk=64, out=None, streams=2, work_size=None):
    """TrimapAgent.forward for every frame: mask-only (trimap/agent.py:35-61) or,
    with ``frames`` and ``bg`` ((3,) colour or [H,W,3] / [N,H,W,3] image), the
    background-gated variant (:63-101) with its per-frame ratio test decided on
    the device."""
    n, h, w = masks.shape
    tri = out if out is not None else torch.empty((n, h, w), dtype=torch.uint8, device=masks.device)
    half = np.array(agent.color_winsize) // 2

    def body(s, e):
        m = masks[s:e]
        if frames is None:
            _trimap_tail(m, agent, out=tri[s:e], work_size=work_size)
            return
        fr = frames[s:e]
        if isinstance(bg, np.ndarray) and bg.ndim == 1:
            hsv = bgr2hsv_pixel(bg)
            fuzzy, counts = ops.fuzzy_count(fr, m, np.clip(hsv - half, 10, 255), np.clip(hsv + half, 10, 255))
        else:
            b = bg[s:e] if bg.ndim == 4 else bg
            bgmask = ops.inrange_image(fr, b, half)
            counts = ops.count_and(m, bgmask)
            fuzzy = ops.mask_and01(m, bgmask)
        flags = ops.ratio_flags(counts, 0.1)       # 0: ensemble, 1: trust mask, 2: empty mask
        # an empty mask is returned as is (all zeros); the plain branch of an all-zero mask is all zeros too
        _trimap_tail(m, agent, fuzzy, flags, out=tri[s:e], work_size=work_size)
    _overlap_chunks(n, chunk, body, streams)
    return tri


def _fused_green_supported(frames, segmasks, cf_agent, trimap_agent):
    """the two-pass green-screen chunk (vu_cf_lowres -> postprocess -> vu_cf_alpha_up_fuzzy -> vu_trimap_bits_packed):
    both agents at the same working resolution, an exact 2x / 4x of it, the 3x3 trimap kernel"""
    n, h, w, _ = frames.shape
    th, tw = get_target_size(h, w, cf_agent.input_long_side)
    return (trimap_agent.input_long_side == cf_agent.input_long_side and trimap_agent.kernelsize == 3 and 0 <= trimap_agent.iters <= 12
            and ops.cf_lowres_supported(h, w, th, tw) and ops.cf_lowres_counts_supported(frames, segmasks, th, tw)
            and ops.cf_up_supported(frames, None, h, w, th, tw, segmasks))


def _fused_green_chunk(fr, sm, cf_agent, trimap_agent, bg_color, alpha_out, tri_out, fg_out=None, bg_out=None):
    """one chunk of green.py:99-114 (+ :125-126 when fg_out / bg_out are given) in five launches and ~7P bytes per frame:
    pass 1 reads the frame and the mask once (HSV, down-scale, mixtures, statistics, early-out counts), the working-
    resolution matte is post-processed in L2, pass 2 writes the full-resolution matte and - from the frame, where the matte
    is non-zero - the fuzzy area and its counts as bits, and the trimap comes out of those bit planes."""
    n, h, w, _ = fr.shape
    th, tw = get_target_size(h, w, cf_agent.input_long_side)
    fg_min, bg_min = max(cf_agent.fg_ncomp) * 5, max(cf_agent.bg_ncomp) * 5
    a_lo, stats, mc = ops.cf_lowres(fr, sm, th, tw, cf_agent.lut3d_dev(), want_mask_counts=True)
    deg = ops.degenerate_flags_from_counts(mc, fg_min, bg_min)
    a_lo = ops.cross_chain(a_lo, [(_lib.DILATE, 2), (_lib.ERODE, 2), (_lib.ERODE, 2), (_lib.DILATE, 2)], stats, 0.8)
    hsv = bgr2hsv_pixel(bg_color)
    half = np.array(trimap_agent.color_winsize) // 2
    res = ops.cf_alpha_up_fuzzy(a_lo, h, w, fr, np.clip(hsv - half, 10, 255), np.clip(hsv + half, 10, 255), alt_src=sm, alt_flags=deg,
                                out=alpha_out, bg_bgr=bg_color if fg_out is not None else None, fg_out=fg_out, bg_out=bg_out)
    _, fzb, mb, counts = res[:4]
    flags = ops.ratio_flags(counts, 0.1)       # 0: ensemble, 1: trust mask, 2: empty mask (its trimap is all zeros either way)
    ops.trimap_bits_packed(mb, fzb, flags, h, w, th, tw, trimap_agent.iters, out=tri_out)


def cf_trimap_clip(frames, segmasks, cf_agent, trimap_agent, bg_color=None, chunk=50, out_alpha=None, out_trimap=None, streams=2, fused=True):
    """BASELINE config 1: ColorFilteringAgent.forward(iters=0) then TrimapAgent.forward(alpha, frame, bg colour) for every
    frame, chunk by chunk.  Chunks bound the temporaries; with ``streams`` = 2 consecutive chunks overlap on two streams and
    fill each other's launch gaps and partial last waves.  ``fused`` (default): the two-pass chunk of _fused_green_chunk
    where the sizes allow it (1080p, 4K), else the stage-by-stage kernels.  Returns alpha, trimap."""
    n, h, w, _ = frames.shape
    dev = frames.device
    alpha = out_alpha if out_alpha is not None else torch.empty((n, h, w), dtype=torch.uint8, device=dev)
    tri = out_trimap if out_trimap is not None else torch.empty((n, h, w), dtype=torch.uint8, device=dev)
    if bg_color is None:
        bg_color = cf_agent.bg_color_bgr()
    use_fused = fused and _fused_green_supported(frames, segmasks, cf_agent, trimap_agent)
    def body(s, e):
        if use_fused:
            _fused_green_chunk(frames[s:e], segmasks[s:e], cf_agent, trimap_agent, bg_color, alpha[s:e], tri[s:e])
            return
        a = cf_predict_clip(frames[s:e], segmasks[s:e], cf_agent, chunk=chunk, out=alpha[s:e])
        trimap_clip(a, trimap_agent, frames[s:e], bg_color, chunk=chunk, out=tri[s:e])
    cf_agent.tables_dev(), cf_agent.lut3d_dev()      # built (once) on the current stream, not on a side stream
    _overlap_chunks(n, chunk, body, streams)
    return alpha, tri


def color_correct_clip(frames, alpha, bg_color, target_long_side=960, mean_exp=0.95, chunk=64, out=None, streams=2):
    """color_correct (imgprocess.py:263-300) over a clip, chunk by chunk (``out`` must not alias ``alpha``)."""
    from .unscreen.utils.imgprocess import get_target_size
    n, h, w, _ = frames.shape
    th, tw = get_target_size(h, w, target_long_side)
    if out is None:
        out = torch.empty_like(alpha)
    _overlap_chunks(n, chunk, lambda s, e: ops.color_correct(frames[s:e], alpha[s:e], bg_color, th, tw, mean_exp, out=out[s:e]), streams)
    return out


def green_clip(frames, segmasks, cf_agent, trimap_agent, chunk=24, bg_color=None, bg_tile=None, color_correct=False, streams=2, fused=True, out=None,
               remove_objects=None, max_objects=16384, tracked=None):
    """the green-screen loop of tools/unscreen/green.py:70-138 without its CNN
    stages (alpha := colour-filter alpha): cf predict -> [remove_invalid_objects, green.py:106-109, when
    ``remove_objects`` = the script's cfg dict is given: the matte the trimap and get_fg see is the cleaned one] -> trimap
    with bg colour -> [color_correct, green.py:120, when asked for] -> bgimg[alpha<128] = frame[...] -> get_fg.
    Like the script, an untracked frame is scored against its segmentation mask (remove_invalid_objects(cfg, alpha,
    segmask)) and a tracked one against its own colour-filter alpha (remove_invalid_objects(cfg, alpha)): ``tracked``
    = per-frame booleans (list, ndarray or device tensor of length n; a device tensor when the call is captured into a
    CUDA graph), None = no frame tracked.  Everything
    stays on the device; a frame with more than ``max_objects`` contours raises after the clip (one read-back).
    Returns alpha, trimap, fg, bg.
    ``bg_color`` ((3,) BGR, host) / ``bg_tile`` ([1,4,3] device) default to the agent's background colour; pass them
    in when the call is captured into a CUDA graph (fetching them synchronises)."""
    n, h, w, _ = frames.shape
    dev = frames.device
    if out is not None:      # (alpha, trimap, fg, bg) of an earlier call: steady-state callers reuse their result buffers
        alpha, tri, fg, bgo = out
    else:
        alpha = torch.empty((n, h, w), dtype=torch.uint8, device=dev)
        tri = torch.empty((n, h, w), dtype=torch.uint8, device=dev)
        fg = torch.empty_like(frames)
        bgo = torch.empty_like(frames)
    if bg_color is None:
        bg_color = cf_agent.bg_color_bgr()
    if bg_tile is None:
        bg_tile = torch.from_numpy(np.tile(bg_color, (1, 4, 1))).to(dev)     # constant background: a 4-pixel periodic image
    use_fused = fused and remove_objects is None and _fused_green_supported(frames, segmasks, cf_agent, trimap_agent)
    statuses = []
    if remove_objects is not None:
        from .unscreen.utils.maskprocess import _score_map_dev
        score_map = _score_map_dev(h, w, remove_objects, dev)
        sal_thr, con_thr = remove_objects['objectremoval']['saliency_thr'], remove_objects['objectremoval']['consensus_thr']
        if tracked is not None:
            tracked = torch.as_tensor(np.asarray(tracked, bool) if not torch.is_tensor(tracked) else tracked, device=dev).bool()
            if tracked.shape != (n,):
                raise ValueError(f"tracked must hold one boolean per frame ({n}), got shape {tuple(tracked.shape)}")
    def body(s, e):
        # every stage writes straight into its slice of the clip-sized results
        if remove_objects is not None:
            a = cf_predict_clip(frames[s:e], segmasks[s:e], cf_agent, chunk=chunk)
            sm = segmasks[s:e] if tracked is None else torch.where(tracked[s:e, None, None], a, segmasks[s:e])
            a, st = ops.remove_invalid_objects(a, sm, score_map, sal_thr, con_thr, max_objects, out=alpha[s:e])
            statuses.append(st)
            trimap_clip(a, trimap_agent, frames[s:e], bg_color, chunk=chunk, out=tri[s:e])
            if color_correct:
                a = color_correct_clip(frames[s:e], a.clone(), bg_color, chunk=chunk, out=alpha[s:e])
            ops.get_fg(frames[s:e], a, bg_tile, _lib.PATCH_ALPHA_LT128, want_bg=True, out=fg[s:e], bg_out=bgo[s:e])
            return
        if use_fused and not color_correct:      # get_fg rides along in the second pass (one BGR2HSV per pixel for both)
            _fused_green_chunk(frames[s:e], segmasks[s:e], cf_agent, trimap_agent, bg_color, alpha[s:e], tri[s:e], fg[s:e], bgo[s:e])
            return
        if use_fused:
            _fused_green_chunk(frames[s:e], segmasks[s:e], cf_agent, trimap_agent, bg_color, alpha[s:e], tri[s:e])
            a = alpha[s:e]
        else:
            a = cf_predict_clip(frames[s:e], segmasks[s:e], cf_agent, chunk=chunk, out=alpha[s:e])
            trimap_clip(a, trimap_agent, frames[s:e], bg_color, chunk=chunk, out=tri[s:e])
        if color_correct:
            a = color_correct_clip(frames[s:e], a.clone(), bg_color, chunk=chunk, out=alpha[s:e])
        ops.get_fg(frames[s:e], a, bg_tile, _lib.PATCH_ALPHA_LT128, want_bg=True, out=fg[s:e], bg_out=bgo[s:e])
    cf_agent.tables_dev(), cf_agent.lut3d_dev()      # built (once) on the current stream, not on a side stream
    _overlap_chunks(n, chunk, body, streams)
    if statuses and int(torch.cat(statuses).max().item()) > max_objects:
        raise RuntimeError(f"green_clip: a frame has more than max_objects = {max_objects} contours; call again with a larger table")
    return alpha, tri, fg, bgo


def replace_clip(fg, alpha, bg, dx=None, dy=None, scale=None, out=None):
    """tools/replace/replace.py:69-76 for a whole clip; ``bg`` is [H,W,3] (shared) or [N,H,W,3].  With ``dx``/``dy``
    and/or ``scale`` the foreground and its mask first go through shift_fg / rescale_fg (:69-72) like in the script;
    without them this is the blend of :74-76 alone (BASELINE config 4).  Whole-clip launches: these kernels fill the
    machine on their own (chunks on two streams were slower, 2.43 against 2.27 ms per 120 frames)."""
    ach = 3 if alpha.ndim == fg.ndim else 1
    if dx is not None or dy is not None:
        fg = ops.shift(fg, dx or 0, dy or 0, 3)
        alpha = ops.shift(alpha, dx or 0, dy or 0, ach)
    if scale is not None:
        fg = ops.rescale_cubic(fg, scale, 3)
        alpha = ops.rescale_cubic(alpha, scale, ach)
    return ops.blend(_lib.BLEND_REPLACE, fg, alpha, bg, out=out)


def bgstep_clip(frames, masks, trimap_agent, thr=25, chunk=24, streams=2, work_size=None, out=None, fused=True):
    """bg_step: exact temporal-median background, then per frame the difference
    gate (bg_offline.py:154-160), mask-only trimap (:166) and get_fg with the
    alpha==0 patch (:171-172), CNN stage skipped (alpha := gated mask).
    Returns background, alpha, trimap, fg.  ``work_size``: the trimap's working
    resolution when ``frames`` is a row tile (see bgstep_clip_tile)."""
    n, h, w, _ = frames.shape
    dev = frames.device
    if out is not None:      # (background, alpha, trimap, fg) of an earlier call, reused
        bg, alpha, tri, fg = out
        ops.temporal_median(frames, out=bg)
    else:
        bg = ops.temporal_median(frames)
        alpha = torch.empty((n, h, w), dtype=torch.uint8, device=dev)
        tri = torch.empty((n, h, w), dtype=torch.uint8, device=dev)
        fg = torch.empty_like(frames)
    th, tw = work_size if work_size is not None else get_target_size(h, w, trimap_agent.input_long_side)
    scale = 2 if (h == 2 * th and w == 2 * tw) else (4 if (h == 4 * th and w == 4 * tw) else 0)
    bits_ok = scale != 0 and tw % 16 == 0 and trimap_agent.kernelsize == 3 and 0 <= trimap_agent.iters <= 12
    def body(s, e):
        # every stage writes straight into its slice of the clip-sized results
        if fused and ops.bgstep_frames_supported(frames[s:e], bg, masks[s:e]) and alpha[s:e].data_ptr() % 16 == 0 and tri[s:e].data_ptr() % 16 == 0:
            # one pass over TMA tiles: gate, matte, get_fg and the trimap's source bits; the trimap from the bits
            a, _, mb = ops.bgstep_frames(frames[s:e], bg, masks[s:e], thr, scale if bits_ok else 0, out_alpha=alpha[s:e], out_fg=fg[s:e])
            if bits_ok:
                ops.trimap_bits_packed(mb, None, None, h, w, th, tw, trimap_agent.iters, out=tri[s:e])
            else:
                trimap_clip(a, trimap_agent, chunk=chunk, out=tri[s:e], work_size=work_size)
            return
        if ops.bgdiff_gate_supported(frames[s:e], bg, masks[s:e]):
            a = ops.bgdiff_gate(frames[s:e], bg, masks[s:e], thr, out=alpha[s:e])
        else:
            a = ops.gate(masks[s:e], ops.dilate(ops.bgdiff_gray(frames[s:e], bg, thr), 4, 2))
            alpha[s:e] = a
        trimap_clip(a, trimap_agent, chunk=chunk, out=tri[s:e], work_size=work_size)
        ops.get_fg(frames[s:e], a, bg, _lib.PATCH_ALPHA_EQ0, out=fg[s:e])
    _overlap_chunks(n, chunk, body, streams)
    return bg, alpha, tri, fg


def bgstep_tile_geometry(h, w, trimap_agent, rank, world):
    """row tile of rank ``rank`` for bgstep_clip_tile on h x w frames: (r0, r1, halo_top, halo_bottom, scale, (th, tw)).
    The working resolution comes from the WHOLE frame (trimap/agent.py:44-46 via get_target_size) and must be an exact
    integer fraction of it (1080p -> 540x960: 2, 4K: 4): only then does a tile that starts on a multiple of the scale
    sample the pixels the whole frame's nearest / bilinear resizes do.  Anything else raises."""
    from . import shard
    th, tw = get_target_size(h, w, trimap_agent.input_long_side)
    scale = h // th if th else 0
    if scale < 1 or h != scale * th or w != scale * tw:
        raise ValueError(f"row-tile sharding needs a working resolution that divides the frame exactly: {h}x{w} -> {th}x{tw}")
    if trimap_agent.kernelsize != 3:
        raise ValueError("row-tile sharding: halo arithmetic is for the 3x3 trimap kernel")
    r0, r1, ht, hb = shard.my_row_tile(h, rank, world, halo=shard.bgstep_halo(scale, trimap_agent.iters), align=scale)
    return r0, r1, ht, hb, scale, (th, tw)


def bgstep_clip_tile(frames, masks, trimap_agent, rank, world, thr=25, chunk=24, rows=None, streams=2, out=None):
    """bgstep_clip on this rank's ROW TILE of the clip (BASELINE config 5: spatial-tile sharding, SURVEY.md section 8e):
    the temporal median of the tile's rows (every pixel is independent), then the per-frame stages on the tile plus a
    halo (shard.bgstep_halo: 28 rows above, 24 below at 4K) read from the local frames, cropped back.  ``frames`` /
    ``masks`` are the WHOLE frames, or -- ``rows`` = (a0, a1, H) -- only rows [a0, a1) of H-row frames, which must
    cover the tile plus its halo (what a rank that holds just its share of the clip passes).  Tile and halo boundaries
    are multiples of the scale (frame size / working size, decided by the WHOLE frame), so the tile's down-scales sample
    the pixels the whole frame's do: the results equal the corresponding rows of bgstep_clip on the whole clip, bit for
    bit.  Returns (r0, r1), background, alpha, trimap, fg for rows [r0, r1) (views of the tile-plus-halo results;
    ``out`` = those tile-plus-halo buffers of an earlier call - ``x._base`` of the returned views - to reuse them)."""
    n, hh, w, _ = frames.shape
    base, h = (rows[0], rows[2]) if rows is not None else (0, hh)
    r0, r1, ht, hb, scale, (th, tw) = bgstep_tile_geometry(h, w, trimap_agent, rank, world)
    a0, a1 = r0 - ht, r1 + hb
    if a0 < base or a1 > base + hh:
        raise ValueError(f"rows [{base}, {base + hh}) do not cover the tile plus halo [{a0}, {a1})")
    ftile = frames[:, a0 - base:a1 - base]
    mtile = masks[:, a0 - base:a1 - base]
    ftile = ftile if ftile.is_contiguous() else ftile.contiguous()
    mtile = mtile if mtile.is_contiguous() else mtile.contiguous()
    bg_t, alpha_t, tri_t, fg_t = bgstep_clip(ftile, mtile, trimap_agent, thr=thr, chunk=chunk, streams=streams,
                                             work_size=((a1 - a0) // scale, tw), out=out)
    lo, hi = ht, ht + (r1 - r0)
    return (r0, r1), bg_t[lo:hi], alpha_t[:, lo:hi], tri_t[:, lo:hi], fg_t[:, lo:hi]
