"""Device-level operators: thin, typed wrappers over the C ABI.

Inputs and outputs are contiguous uint8 CUDA tensors (torch is used for device
memory and streams only).  Images are [H,W,3] or [N,H,W,3] (BGR), masks [H,W]
or [N,H,W].  Every function enqueues on torch's current stream and returns
device tensors; nothing synchronises.
"""
import ctypes

import numpy as np
import torch

from . import _lib
from ._lib import check, i3, lib

u8 = torch.uint8


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _p(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else ctypes.c_void_p(0)


def _dev(t, dtype=u8):
    if not (isinstance(t, torch.Tensor) and t.is_cuda and t.dtype == dtype):
        raise TypeError(f"expected a CUDA {dtype} tensor, got {type(t)} {getattr(t, 'dtype', None)} {getattr(t, 'device', None)}")
    return t if t.is_contiguous() else t.contiguous()


def _img(t):
    t = _dev(t)
    if t.ndim not in (3, 4) or t.shape[-1] != 3:
        raise ValueError(f"expected [H,W,3] or [N,H,W,3], got {tuple(t.shape)}")
    return t


def _mask(t):
    t = _dev(t)
    if t.ndim not in (2, 3):
        raise ValueError(f"expected [H,W] or [N,H,W], got {tuple(t.shape)}")
    return t


# ---- colour ---------------------------------------------------------------

def bgr2hsv(x):
    x = _img(x)
    out = torch.empty_like(x)
    check(lib().vu_bgr2hsv_u8(_p(x), _p(out), x.numel() // 3, _stream()))
    return out


def hsv2bgr(x):
    x = _img(x)
    out = torch.empty_like(x)
    check(lib().vu_hsv2bgr_u8(_p(x), _p(out), x.numel() // 3, _stream()))
    return out


def bgr2gray(x):
    x = _img(x)
    out = torch.empty(x.shape[:-1], dtype=u8, device=x.device)
    check(lib().vu_bgr2gray_u8(_p(x), _p(out), x.numel() // 3, _stream()))
    return out


def inrange_color(x, lo, hi):
    """0/1 mask of lo <= HSV(x) <= hi (inclusive, per channel)."""
    x = _img(x)
    out = torch.empty(x.shape[:-1], dtype=u8, device=x.device)
    check(lib().vu_inrange_color(_p(x), x.numel() // 3, i3(lo), i3(hi), _p(out), _stream()))
    return out


def inrange_image(x, bg, half):
    """0/1 mask of clamp(HSV(bg)-half,10,255) <= HSV(x) <= clamp(HSV(bg)+half,10,255)."""
    x, bg = _img(x), _img(bg)
    if bg.shape[-3:] != x.shape[-3:]:
        raise ValueError("background image must have the frame's H,W")
    if bg.ndim == 4 and bg.shape != x.shape:
        raise ValueError("batched background must match the frames' shape")
    out = torch.empty(x.shape[:-1], dtype=u8, device=x.device)
    check(lib().vu_inrange_image(_p(x), _p(bg), x.numel() // 3, bg.numel() // 3, i3(half), _p(out), _stream()))
    return out


# ---- morphology / resize ----------------------------------------------------

CROSS_MAX_PASSES = 12


def morph(x, ksize, iters, op):
    """cv2.dilate / cv2.erode with MORPH_ELLIPSE(ksize, ksize), `iters` iterations."""
    if int(ksize) == 3 and int(iters) <= CROSS_MAX_PASSES:
        return cross_chain(x, [(op, iters)])
    x = _mask(x)
    n = 1 if x.ndim == 2 else x.shape[0]
    h, w = x.shape[-2:]
    out = torch.empty_like(x)
    ws_bytes = int(lib().vu_morph_workspace_bytes(n, h, w, int(ksize), int(iters)))   # 0 unless the iterations need several launches
    ws = torch.empty(ws_bytes, dtype=u8, device=x.device) if ws_bytes else None
    check(lib().vu_morph_u8(_p(x), _p(out), n, h, w, int(ksize), int(iters), op, _p(ws), ws_bytes, _stream()))
    return out


def cross_chain(x, segments, stats=None, thr_ratio=0.8):
    """chain of (op, iters) segments of the 3x3 cross in one kernel; with
    ``stats`` ([n,2] int64 sum/count) the colour-filter threshold is applied on load."""
    x = _mask(x)
    n = 1 if x.ndim == 2 else x.shape[0]
    h, w = x.shape[-2:]
    segs = [(int(o), int(i)) for o, i in segments]
    if not 1 <= len(segs) <= 4 or sum(i for _, i in segs) > CROSS_MAX_PASSES:
        raise ValueError("cross_chain: 1..4 segments, at most 12 passes")
    segs += [(0, 0)] * (4 - len(segs))
    ops_a = (ctypes.c_int32 * 4)(*[o for o, _ in segs])
    it_a = (ctypes.c_int32 * 4)(*[i for _, i in segs])
    out = torch.empty_like(x)
    sp = _p(_dev(stats, torch.int64)) if stats is not None else ctypes.c_void_p(0)
    check(lib().vu_cross_chain_u8(_p(x), _p(out), n, h, w, len(segments), ops_a, it_a, sp, float(thr_ratio), _stream()))
    return out


def trimap_core(mask_lo, iters):
    """classify(dilate^iters, erode^iters) of the 3x3 cross in one kernel (trimap/agent.py:53-58)."""
    x = _mask(mask_lo)
    n = 1 if x.ndim == 2 else x.shape[0]
    h, w = x.shape[-2:]
    out = torch.empty_like(x)
    check(lib().vu_trimap_core_u8(_p(x), _p(out), n, h, w, int(iters), _stream()))
    return out


def trimap_bits_supported(masks, th, tw, iters, fuzzy=None):
    h, w = masks.shape[-2:]
    exact = (h == 2 * th and w == 2 * tw) or (h == 4 * th and w == 4 * tw)
    al = masks.data_ptr() % 16 == 0 and (fuzzy is None or fuzzy.data_ptr() % 16 == 0)
    return exact and tw % 4 == 0 and 0 <= int(iters) <= 12 and al


def trimap_bits(masks, th, tw, iters, fuzzy=None, flags=None, out=None):
    """the trimap tail of trimap/agent.py:52-60 (+ the ensemble's :97 / :100 with ``fuzzy`` and ``flags``) in bit logic for
    exact 2x / 4x working resolutions: masks [N,H,W] (or [H,W]) -> trimaps of the same shape."""
    x = _mask(masks)
    n = 1 if x.ndim == 2 else x.shape[0]
    h, w = x.shape[-2:]
    out = _out(out, x.shape, x.device)
    ws_bytes = int(lib().vu_trimap_bits_workspace_bytes(n, int(th), int(tw)))
    ws = torch.empty(ws_bytes, dtype=u8, device=x.device)
    fz = _p(_dev(fuzzy)) if fuzzy is not None else ctypes.c_void_p(0)
    fl = _p(_dev(flags)) if flags is not None else ctypes.c_void_p(0)
    check(lib().vu_trimap_bits(_p(x), fz, fl, n, h, w, int(th), int(tw), int(iters), _p(out), _p(ws), ws_bytes, _stream()))
    return out


def cf_up_supported(frames, alpha_lo, h, w, th, tw, *others):
    """vu_cf_alpha_up_fuzzy / vu_trimap_bits_packed: exact 2x / 4x working resolution, tw % 16 == 0, 16-byte aligned clips"""
    exact = (h == 2 * th and w == 2 * tw) or (h == 4 * th and w == 4 * tw)
    return exact and tw % 16 == 0 and all(t is None or t.data_ptr() % 16 == 0 for t in (frames, alpha_lo) + others)


def cf_alpha_up_fuzzy(alpha_lo, h, w, frames, lo, hi, alt_src=None, alt_flags=None, out=None, bg_bgr=None, fg_out=None, bg_out=None):
    """colorfiltering/agent.py:342 + trimap/agent.py:84-94 (+ green.py:125-126 with ``bg_bgr``) in one pass, see
    vu_cf_alpha_up_fuzzy.  -> alpha [n,h,w], fuzzy bits [n,h,w/8], mask bits [n,th,tw/8], counts [n,2] (+ fg, bg)."""
    alpha_lo, frames = _mask(alpha_lo), _img(frames)
    n = 1 if alpha_lo.ndim == 2 else alpha_lo.shape[0]
    th, tw = alpha_lo.shape[-2:]
    dev = alpha_lo.device
    alpha = _out(out, (h, w) if alpha_lo.ndim == 2 else (n, h, w), dev)
    fzb = torch.empty((n, h, w // 8), dtype=u8, device=dev)
    mb = torch.empty((n, th, tw // 8), dtype=u8, device=dev)
    counts = torch.empty((n, 2), dtype=torch.int64, device=dev)
    col = None
    if bg_bgr is not None:
        col = np.ascontiguousarray(np.asarray(bg_bgr, dtype=np.uint8).reshape(3))
        fg_out = _out(fg_out, frames.shape, dev)
        bg_out = _out(bg_out, frames.shape, dev)
    check(lib().vu_cf_alpha_up_fuzzy(_p(alpha_lo), n, th, tw, int(h), int(w), _p(alt_src), _p(alt_flags), _p(frames), i3(lo), i3(hi), _p(alpha),
                                     _p(fzb), _p(mb), _p(counts), col.ctypes.data if col is not None else None, _p(fg_out), _p(bg_out), _stream()))
    return (alpha, fzb, mb, counts) + ((fg_out, bg_out) if col is not None else ())


def trimap_bits_packed(mask_bits, fuzzy_bits, flags, h, w, th, tw, iters, out=None):
    """the trimap tail from the bit planes of cf_alpha_up_fuzzy (vu_trimap_bits_packed) -> trimaps [n,h,w]"""
    n = mask_bits.shape[0]
    out = _out(out, (n, h, w), mask_bits.device)
    ws_bytes = int(lib().vu_trimap_bits_workspace_bytes(n, int(th), int(tw)))
    ws = torch.empty(ws_bytes, dtype=u8, device=mask_bits.device)
    check(lib().vu_trimap_bits_packed(_p(_dev(mask_bits)), _p(fuzzy_bits), _p(flags), n, int(h), int(w), int(th), int(tw), int(iters), _p(out),
                                      _p(ws), ws_bytes, _stream()))
    return out


def dilate(x, ksize, iters):
    return morph(x, ksize, iters, _lib.DILATE)


def erode(x, ksize, iters):
    return morph(x, ksize, iters, _lib.ERODE)


def _resize(fn, x, dh, dw, channels):
    x = _dev(x)
    if channels == 3:
        x = _img(x)
        n = 1 if x.ndim == 3 else x.shape[0]
        sh, sw = x.shape[-3:-1]
        shape = (dh, dw, 3) if x.ndim == 3 else (n, dh, dw, 3)
    else:
        x = _mask(x)
        n = 1 if x.ndim == 2 else x.shape[0]
        sh, sw = x.shape[-2:]
        shape = (dh, dw) if x.ndim == 2 else (n, dh, dw)
    out = torch.empty(shape, dtype=u8, device=x.device)
    check(fn(_p(x), n, sh, sw, channels, _p(out), int(dh), int(dw), _stream()))
    return out


def resize_linear_mask(x, dh, dw):
    x = _mask(x)
    sh, sw = x.shape[-2:]
    if (sh, sw) == (dh, dw) or (sh == 2 * dh and sw == 2 * dw):
        return _resize(lib().vu_resize_linear_u8, x, dh, dw, 1)   # copy / cv2's silent INTER_AREA
    return resize_up(x, dh, dw)


def _out(out, shape, device):
    """the caller's output tensor (a contiguous uint8 CUDA tensor of the right shape: e.g. a slice of a clip-sized result,
    so that chunked pipelines do not copy their chunks) or a fresh one."""
    if out is None:
        return torch.empty(shape, dtype=u8, device=device)
    if tuple(out.shape) != tuple(shape) or out.dtype != u8 or not out.is_cuda or not out.is_contiguous():
        raise ValueError(f"out must be a contiguous CUDA uint8 tensor of shape {tuple(shape)}")
    return out


def resize_up(x, dh, dw, mode=0, fuzzy=None, flags=None, alt_src=None, alt_flags=None, out=None):
    """cv2.resize (bilinear) of masks with fused epilogues (see vu_resize_up_u8)."""
    x = _mask(x)
    n = 1 if x.ndim == 2 else x.shape[0]
    sh, sw = x.shape[-2:]
    out = _out(out, (dh, dw) if x.ndim == 2 else (n, dh, dw), x.device)
    check(lib().vu_resize_up_u8(_p(x), n, sh, sw, _p(out), int(dh), int(dw), int(mode), _p(fuzzy), _p(flags), _p(alt_src), _p(alt_flags),
                                _stream()))
    return out


def cf_lowres(frames, masks, th, tw, lut3d, want_mask_counts=False):
    """fused BGR2HSV + down-scale + tabulated mixtures + postprocess statistics; -> (alpha_lo, stats[, mask_counts]).
    ``want_mask_counts`` (see cf_lowres_counts_supported): also [n,2] = (#(mask > 128), #(mask < 128)) per frame."""
    frames, masks, lut3d = _img(frames), _mask(masks), _dev(lut3d)
    n = 1 if frames.ndim == 3 else frames.shape[0]
    h, w = frames.shape[-3:-1]
    alpha = torch.empty((th, tw) if frames.ndim == 3 else (n, th, tw), dtype=u8, device=frames.device)
    stats = torch.empty((n, 2), dtype=torch.int64, device=frames.device)
    mc = torch.empty((n, 2), dtype=torch.int64, device=frames.device) if want_mask_counts else None
    check(lib().vu_cf_lowres(_p(frames), _p(masks), n, h, w, int(th), int(tw), _p(lut3d), _p(alpha), _p(stats), _p(mc), _stream()))
    return (alpha, stats, mc) if want_mask_counts else (alpha, stats)


def cf_lowres_counts_supported(frames, masks, th, tw):
    h, w = frames.shape[-3:-1]
    exact = (h == 2 * th and w == 2 * tw and tw % 8 == 0) or (h == 4 * th and w == 4 * tw and tw % 4 == 0)
    return exact and w % 16 == 0 and frames.data_ptr() % 16 == 0 and masks.data_ptr() % 16 == 0


def degenerate_flags_from_counts(counts2, fg_min, bg_min):
    """per-frame early-out flags of ColorFilteringAgent.forward from [n,2] (#(mask > 128), #(mask < 128))"""
    c = _dev(counts2, torch.int64)
    n = c.shape[0]
    flags = torch.empty(n, dtype=u8, device=c.device)
    second = ctypes.c_void_p(c.data_ptr() + 8)
    check(lib().vu_cf_degenerate_flags(_p(c), second, n, 2, int(fg_min), int(bg_min), _p(flags), _stream()))
    return flags


def cf_lowres_supported(h, w, th, tw):
    return ((h == 2 * th and w == 2 * tw) or (h == 4 * th and w == 4 * tw)) and w % 4 == 0 and tw % 2 == 0


def fuzzy_count(frames, alpha, lo, hi):
    """-> (fuzzy01 [n,h,w], counts [n,2] = (#fuzzy, #alpha>0)); trimap/agent.py:90-94"""
    frames, alpha = _img(frames), _mask(alpha)
    n = 1 if frames.ndim == 3 else frames.shape[0]
    fuzzy = torch.empty_like(alpha)
    counts = torch.empty((n, 2), dtype=torch.int64, device=frames.device)
    check(lib().vu_fuzzy_count(_p(frames), _p(alpha), n, alpha.numel() // n, i3(lo), i3(hi), _p(fuzzy), _p(counts), _stream()))
    return fuzzy, counts


def trimap_src_lo(mask, th, tw, fuzzy=None, flags=None):
    mask = _mask(mask)
    n = 1 if mask.ndim == 2 else mask.shape[0]
    h, w = mask.shape[-2:]
    out = torch.empty((th, tw) if mask.ndim == 2 else (n, th, tw), dtype=u8, device=mask.device)
    check(lib().vu_trimap_src_lo(_p(mask), _p(fuzzy), _p(flags), n, h, w, int(th), int(tw), _p(out), _stream()))
    return out


def resize_linear_image(x, dh, dw):
    return _resize(lib().vu_resize_linear_u8, x, dh, dw, 3)


def resize_linear(x, dh, dw):
    """cv2.resize(x, (dw, dh)) of an image [H,W,3] or a single-channel [H,W] array, any ratio"""
    return _resize(lib().vu_resize_linear_u8, x, dh, dw, 3 if x.ndim == 3 else 1)


def resize_nearest_mask(x, dh, dw):
    return _resize(lib().vu_resize_nearest_u8, x, dh, dw, 1)


def resize_nearest_image(x, dh, dw):
    return _resize(lib().vu_resize_nearest_u8, x, dh, dw, 3)


# ---- geometric pre-steps of the replacement path ------------------------------

def _geom_shape(x, channels):
    """(n, h, w) of an image [H,W,3] / clip [N,H,W,3] (channels 3) or a mask [H,W] / [N,H,W] (channels 1)."""
    if channels == 3:
        x = _img(x)
        return x, (1 if x.ndim == 3 else x.shape[0]), x.shape[-3], x.shape[-2]
    if channels != 1:
        raise ValueError("channels must be 1 or 3")
    x = _mask(x)
    return x, (1 if x.ndim == 2 else x.shape[0]), x.shape[-2], x.shape[-1]


def shift(x, dx, dy, channels=3):
    """shift_fg (imgprocess.py:55-64): cv2.warpAffine translation by (dx, dy), zero border."""
    x, n, h, w = _geom_shape(_dev(x), channels)
    out = torch.empty_like(x)
    check(lib().vu_shift_u8(_p(x), _p(out), n, h, w, channels, float(dx), float(dy), _stream()))
    return out


def rescale_cubic(x, factor, channels=3):
    """rescale_fg (imgprocess.py:40-52): bicubic up-scale by ``factor`` and centre crop to the input size."""
    x, n, h, w = _geom_shape(_dev(x), channels)
    out = torch.empty_like(x)
    check(lib().vu_rescale_cubic_u8(_p(x), _p(out), n, h, w, channels, float(factor), _stream()))
    return out


def color_correct(frames, alpha, bg_color, th, tw, mean_exp=0.95, out=None):
    """color_correct (imgprocess.py:263-300) for an image [H,W,3] + alpha [H,W] or a clip [N,H,W,3] + [N,H,W]:
    alpha scaled by the normalised Lab chroma distance to ``bg_color`` (3 uint8 values, host side) computed at the
    working resolution th x tw."""
    frames, alpha = _img(frames), _mask(alpha)
    n = 1 if frames.ndim == 3 else frames.shape[0]
    h, w = frames.shape[-3], frames.shape[-2]
    if tuple(alpha.shape[-2:]) != (h, w) or alpha.numel() != n * h * w:
        raise ValueError(f"alpha {tuple(alpha.shape)} does not match frames {tuple(frames.shape)}")
    col = np.ascontiguousarray(np.asarray(bg_color, dtype=np.uint8).reshape(3))
    ws = torch.empty(lib().vu_color_correct_workspace_bytes(n, th, tw), dtype=u8, device=frames.device)
    out = _out(out, alpha.shape, alpha.device)
    rc = lib().vu_color_correct_frames(_p(frames), _p(alpha), n, h, w, int(th), int(tw), col.ctypes.data, float(mean_exp), _p(out), _p(ws),
                                       ws.numel(), _stream())
    if rc != _lib.ERR_UNSUPPORTED:      # exact 2x / 4x working resolution: the down-scale is fused into the first kernel
        check(rc)
        return out
    frames_lo = resize_linear_image(frames, th, tw)
    alpha_lo = resize_linear_mask(alpha, th, tw)
    check(lib().vu_color_correct(_p(frames_lo), _p(alpha_lo), _p(alpha), n, h, w, int(th), int(tw), col.ctypes.data, float(mean_exp), _p(out),
                                 _p(ws), ws.numel(), _stream()))
    return out


# ---- reductions / mask algebra ----------------------------------------------

def _items(x, item_ndim):
    n = 1 if x.ndim == item_ndim else x.shape[0]
    return n, x.numel() // max(n, 1)


def count_cmp(x, op, thr, item_ndim=2):
    """per-item counts (int64 device tensor [n]) of x <op> thr."""
    x = _dev(x)
    n, per = _items(x, item_ndim)
    out = torch.empty(n, dtype=torch.int64, device=x.device)
    check(lib().vu_count_cmp_u8(_p(x), n, per, op, int(thr), _p(out), _stream()))
    return out


def count_and(a, b, item_ndim=2):
    """[n,2] int64: (#{a>0 & b>0}, #{a>0}) per item."""
    a, b = _dev(a), _dev(b)
    n, per = _items(a, item_ndim)
    out = torch.empty((n, 2), dtype=torch.int64, device=a.device)
    check(lib().vu_count_and_u8(_p(a), _p(b), n, per, _p(out), _stream()))
    return out


def _binary(fn, a, b):
    a, b = _dev(a), _dev(b)
    if a.shape != b.shape:
        raise ValueError("shape mismatch")
    out = torch.empty_like(a)
    check(fn(_p(a), _p(b), _p(out), a.numel(), _stream()))
    return out


def mask_clear_where(a, b):
    return _binary(lib().vu_mask_clear_where, a, b)


def mask_set128_where(a, b):
    return _binary(lib().vu_mask_set128_where, a, b)


def mask_and01(a, b):
    return _binary(lib().vu_mask_and01, a, b)


def trimap_classify(dilated, eroded):
    return _binary(lib().vu_trimap_classify, dilated, eroded)


def trimap_snap(a):
    a = _dev(a)
    out = torch.empty_like(a)
    check(lib().vu_trimap_snap(_p(a), a.numel(), _p(out), _stream()))
    return out


def gate(mask, g):
    mask, g = _dev(mask), _dev(g)
    out = torch.empty_like(mask)
    check(lib().vu_gate(_p(mask), _p(g), mask.numel(), _p(out), _stream()))
    return out


def bgdiff_gate_supported(frames, bg, masks):
    return frames.shape[-2] % 4 == 0 and all(t.data_ptr() % 8 == 0 for t in (frames, bg, masks))


def bgdiff_gate(frames, bg, masks, thr, out=None):
    """mask * (dilate_mask(g, 4, 2) // 255), g = thresholded BGR2GRAY(|frame - bg|), fused and bit-packed
    (tools/unscreen/bg.py:85-92 == bg_offline.py:154-160); frames [N,H,W,3] or [H,W,3], bg [H,W,3] or [N,H,W,3]."""
    frames, bg, masks = _img(frames), _img(bg), _dev(masks)
    h, w = frames.shape[-3], frames.shape[-2]
    n = frames.numel() // (h * w * 3)
    nb = bg.numel() // (h * w * 3)
    out = _out(out, masks.shape, masks.device)
    check(lib().vu_bgdiff_gate(_p(frames), _p(bg), _p(masks), n, h, w, nb, int(thr), _p(out), _stream()))
    return out


def bgstep_frames_supported(frames, bg, masks):
    return frames.shape[-2] % 16 == 0 and all(t.data_ptr() % 16 == 0 for t in (frames, bg, masks))


def bgstep_frames(frames, bg, masks, thr, scale=0, out_alpha=None, out_fg=None):
    """difference gate + get_fg(patch alpha == 0) (+ the trimap's source bits for an exact ``scale`` = 2 / 4) in one pass over
    TMA tiles (vu_bgstep_frames; bg_offline.py:154-160, :171-172).  -> alpha, fg, mask_bits (None when scale == 0)."""
    frames, bg, masks = _img(frames), _img(bg), _dev(masks)
    h, w = frames.shape[-3], frames.shape[-2]
    n = frames.numel() // (h * w * 3)
    nb = bg.numel() // (h * w * 3)
    alpha = _out(out_alpha, masks.shape, masks.device)
    fg = _out(out_fg, frames.shape, frames.device)
    mb = torch.empty((n, h // scale, w // scale // 8), dtype=u8, device=frames.device) if scale else None
    check(lib().vu_bgstep_frames(_p(frames), _p(bg), _p(masks), n, h, w, nb, int(thr), _p(alpha), _p(fg), _p(mb), int(scale), _stream()))
    return alpha, fg, mb


def sub_wrap(a, b):
    a, b = _dev(a), _dev(b)
    out = torch.empty_like(a)
    check(lib().vu_sub_wrap_u8(_p(a), _p(b), a.numel(), _p(out), _stream()))
    return out


def binarise(a, thr=128):
    a = _dev(a)
    out = torch.empty_like(a)
    check(lib().vu_binarise(_p(a), a.numel(), int(thr), _p(out), _stream()))
    return out


# ---- colour filtering ---------------------------------------------------------

def cf_alpha(hsv, luts):
    hsv = _img(hsv)
    luts = _dev(luts, torch.float32)
    assert luts.numel() == 6 * 256
    out = torch.empty(hsv.shape[:-1], dtype=u8, device=hsv.device)
    check(lib().vu_cf_alpha_u8(_p(hsv), hsv.numel() // 3, _p(luts), _p(out), _stream()))
    return out


def cf_build_lut3d(luts):
    luts = _dev(luts, torch.float32)
    assert luts.numel() == 6 * 256
    out = torch.empty((180, 256, 256), dtype=u8, device=luts.device)
    check(lib().vu_cf_build_lut3d(_p(luts), _p(out), _stream()))
    return out


def cf_alpha_lut3d(hsv, lut3d):
    hsv, lut3d = _img(hsv), _dev(lut3d)
    assert lut3d.numel() == 180 * 256 * 256
    out = torch.empty(hsv.shape[:-1], dtype=u8, device=hsv.device)
    check(lib().vu_cf_alpha_lut3d_u8(_p(hsv), hsv.numel() // 3, _p(lut3d), _p(out), _stream()))
    return out


def cf_threshold_stats(alpha, mask):
    """per item {sum, count} of alpha over (alpha > 128 and mask > 0)."""
    alpha, mask = _mask(alpha), _mask(mask)
    n, per = _items(alpha, 2)
    stats = torch.empty((n, 2), dtype=torch.int64, device=alpha.device)
    check(lib().vu_cf_threshold_stats(_p(alpha), _p(mask), n, per, _p(stats), _stream()))
    return stats


def cf_postprocess(alpha, mask, thr_ratio=0.8):
    """ColorFilteringAgent.postprocess (agent.py:259-283): adaptive threshold then
    d2,e2,e2,d2, the threshold fused into the morphology kernel's load."""
    stats = cf_threshold_stats(alpha, mask)
    return cross_chain(alpha, [(_lib.DILATE, 2), (_lib.ERODE, 2), (_lib.ERODE, 2), (_lib.DILATE, 2)], stats, thr_ratio)


def cf_threshold(alpha, mask, thr_ratio=0.8):
    """postprocess step 1 (adaptive threshold), per item."""
    alpha, mask = _mask(alpha), _mask(mask)
    n, per = _items(alpha, 2)
    stats = torch.empty((n, 2), dtype=torch.int64, device=alpha.device)
    check(lib().vu_cf_threshold_stats(_p(alpha), _p(mask), n, per, _p(stats), _stream()))
    out = torch.empty_like(alpha)
    check(lib().vu_cf_threshold_apply(_p(alpha), n, per, _p(stats), float(thr_ratio), _p(out), _stream()))
    return out


# ---- compositing ----------------------------------------------------------------

def _check_bg(bg, img, what):
    """a background the kernels index correctly: the image's own shape, one [H,W,3] image under a clip, or the constant
    tile ([1,4,3] / [1,1,3]: the caller's four pixels are one colour).  Anything else would wrap around silently."""
    if tuple(bg.shape) == tuple(img.shape) or (img.ndim == 4 and tuple(bg.shape) == tuple(img.shape[1:])):
        return
    if bg.ndim == 3 and bg.shape[0] == 1 and bg.shape[1] in (1, 4) and img.shape[-3:-1] != (1, 4):
        return
    raise ValueError(f"{what}: background {tuple(bg.shape)} does not match the image {tuple(img.shape)}")


def get_fg(frame, alpha, bg, patch=_lib.PATCH_NONE, want_bg=False, out=None, bg_out=None):
    frame, alpha, bg = _img(frame), _mask(alpha), _img(bg)
    if alpha.shape != frame.shape[:-1]:
        raise ValueError("alpha must have the frame's [N,]H,W")
    _check_bg(bg, frame, "get_fg")
    fg = _out(out, frame.shape, frame.device)
    bgo = _out(bg_out, frame.shape, frame.device) if want_bg else None
    check(lib().vu_get_fg(_p(frame), _p(alpha), _p(bg), frame.numel() // 3, bg.numel() // 3, patch, _p(fg), _p(bgo), _stream()))
    return (fg, bgo) if want_bg else fg


def get_bg(alpha, bg):
    alpha, bg = _mask(alpha), _img(bg)
    out = torch.empty_like(bg)
    check(lib().vu_get_bg(_p(alpha), _p(bg), bg.numel() // 3, _p(out), _stream()))
    return out


def blend(mode, fg, alpha, bg=None, out=None):
    fg, alpha = _img(fg), _dev(alpha)
    ac = 3 if alpha.shape == fg.shape else 1
    if ac == 1 and alpha.shape != fg.shape[:-1]:
        raise ValueError("alpha must be [N,]H,W or the image's shape")
    if bg is not None:
        bg = _img(bg)
        _check_bg(bg, fg, "blend")
    out = _out(out, fg.shape, fg.device)
    check(lib().vu_blend(mode, _p(fg), _p(alpha), ac, _p(bg), fg.numel() // 3, (bg.numel() // 3) if bg is not None else 0, _p(out), _stream()))
    return out


def fuse_bg(bg, bg_always, beta):
    import numpy as np
    bg, bg_always = _img(bg), _img(bg_always)
    out = torch.empty_like(bg)
    b = float(np.float32(beta))
    omb = float(np.float32(1 - beta))
    check(lib().vu_fuse_bg(_p(bg), _p(bg_always), bg.numel() // 3, bg_always.numel() // 3, b, omb, _p(out), _stream()))
    return out


def bgdiff_gray(frame, bg, thr):
    frame, bg = _img(frame), _img(bg)
    out = torch.empty(frame.shape[:-1], dtype=u8, device=frame.device)
    check(lib().vu_bgdiff_gray(_p(frame), _p(bg), frame.numel() // 3, bg.numel() // 3, int(thr), _p(out), _stream()))
    return out


# ---- temporal ---------------------------------------------------------------------

def temporal_median(frames, out=None):
    frames = _dev(frames)
    n = frames.shape[0]
    m = frames.numel() // n
    if out is None:
        out = torch.empty(frames.shape[1:], dtype=u8, device=frames.device)
    ws_bytes = int(lib().vu_temporal_median_workspace_bytes(n, m))
    if ws_bytes:
        ws = torch.empty(ws_bytes, dtype=u8, device=frames.device)
        check(lib().vu_temporal_median_u8_ws(_p(frames), n, m, _p(out), _p(ws), ws_bytes, _stream()))
    else:
        check(lib().vu_temporal_median_u8(_p(frames), n, m, _p(out), _stream()))
    return out


def masked_temporal_mean(frames, masks_dilated, min_count=10):
    frames, masks_dilated = _img(frames), _mask(masks_dilated)
    n, h, w, _ = frames.shape
    bg = torch.empty((h, w, 3), dtype=u8, device=frames.device)
    always = torch.empty((h, w), dtype=u8, device=frames.device)
    check(lib().vu_masked_temporal_mean(_p(frames), _p(masks_dilated), n, h * w, int(min_count), _p(bg), _p(always), _stream()))
    return bg, always


def masked_temporal_mean_raw(frames, masks, ksize=3, iters=2, min_count=10):
    """bg_offline.py:106-125 from the raw masks: dilate_mask(mask, ksize, iters) then the masked mean; for the script's
    (3, 2) the dilation is fused into the mean as bit-plane logic (vu_masked_temporal_mean_dilate32)."""
    frames, masks = _img(frames), _mask(masks)
    n, h, w, _ = frames.shape
    if (ksize, iters) == (3, 2):
        bg = torch.empty((h, w, 3), dtype=u8, device=frames.device)
        always = torch.empty((h, w), dtype=u8, device=frames.device)
        rc = lib().vu_masked_temporal_mean_dilate32(_p(frames), _p(masks), n, h, w, int(min_count), _p(bg), _p(always), _stream())
        if rc != _lib.ERR_UNSUPPORTED:
            check(rc)
            return bg, always
    return masked_temporal_mean(frames, dilate(masks, ksize, iters), min_count)


MEDIAN_ACCUM_MAX_FRAMES = 65535      # 16-bit histogram counters
MEAN_ACCUM_MAX_FRAMES = 16000000     # 32-bit sums of bytes


class TemporalMedianAccumulator:
    """The exact temporal median of a clip that arrives in chunks: ``add`` any number of batches [k, *frame_shape], in any
    order, then ``result()`` is ``temporal_median`` of all of them together, byte for byte.  The state is 512 bytes per frame
    byte (3.2 GB at 1080p, 12.7 GB at 4K) whatever the clip length; at most 65535 frames.  Every call enqueues on the
    current stream and neither allocates device memory (except ``result``'s output) nor synchronises, so an ``add`` can
    run on a side stream or inside a CUDA graph.  A captured add always accumulates into the state, whatever ``.n`` was at
    capture.  ``.n`` is counted on the host when ``add`` is called, so it does not see replays, and the 65535-frame limit
    is not checked for them: after replaying a captured add of k frames r times, add r * k to ``.n`` (a plain attribute)
    before ``result()``, and keep the total at most 65535.  Each add reads and writes the whole state: chunks of hundreds
    of frames."""

    def __init__(self, frame_shape, device=None):
        self.frame_shape = tuple(int(s) for s in frame_shape)
        self.m = int(np.prod(self.frame_shape, dtype=np.int64))
        self.device = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
        nbytes = int(lib().vu_median_accum_bytes(self.m))
        self.state = torch.empty(max(nbytes, 16), dtype=u8, device=self.device)
        self.reset()

    def reset(self):
        check(lib().vu_median_accum_reset(_p(self.state), self.m, _stream()))
        self.n = 0

    def add(self, frames):
        frames = _dev(frames)
        if tuple(frames.shape[1:]) != self.frame_shape:
            raise ValueError(f"expected frames [k, {self.frame_shape}], got {tuple(frames.shape)}")
        k = frames.shape[0]
        if k == 0:
            return self
        rc = lib().vu_median_accum_add_u8(_p(self.state), self.m, _p(frames), k, self.n, _stream())
        if rc != _lib.VU_OK and self.n + k > MEDIAN_ACCUM_MAX_FRAMES:     # refused, the state untouched
            raise _lib.VuError(f"the median accumulator holds at most {MEDIAN_ACCUM_MAX_FRAMES} frames: {self.n} + {k}")
        check(rc)
        self.n += k
        return self

    def result(self, out=None):
        if out is None:
            out = torch.empty(self.frame_shape, dtype=u8, device=self.device)
        elif not (out.is_cuda and out.dtype == u8 and out.is_contiguous() and out.numel() == self.m):
            raise ValueError(f"out must be a contiguous CUDA uint8 tensor of {self.m} bytes")
        check(lib().vu_median_accum_finish_u8(_p(self.state), self.m, self.n, _p(out), _stream()))
        return out


class MaskedMeanAccumulator:
    """bg_offline.py:106-125 for a clip that arrives in chunks: ``add(frames [k,h,w,3], masks [k,h,w])`` with the RAW masks
    (dilated by dilate_mask(mask, ksize, iters) like ``masked_temporal_mean_raw``), in any chunking and order; ``result()``
    returns (bg [h,w,3], mask_always [h,w]), byte for byte those of ``masked_temporal_mean_raw`` on the whole clip.  16 bytes
    of state per pixel.  Enqueues on the current stream; nothing synchronises."""

    def __init__(self, h, w, ksize=3, iters=2, min_count=10, device=None):
        self.h, self.w = int(h), int(w)
        self.ksize, self.iters, self.min_count = int(ksize), int(iters), int(min_count)
        self.device = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
        self.state = torch.empty(int(lib().vu_masked_mean_accum_bytes(self.h, self.w)), dtype=u8, device=self.device)
        self.reset()

    def reset(self):
        check(lib().vu_masked_mean_accum_reset(_p(self.state), self.h, self.w, _stream()))
        self.n = 0

    def add(self, frames, masks):
        frames, masks = _img(frames), _mask(masks)
        k = frames.shape[0]
        if frames.shape != (k, self.h, self.w, 3) or masks.shape != (k, self.h, self.w):
            raise ValueError(f"expected frames [k,{self.h},{self.w},3] and masks [k,{self.h},{self.w}], got {tuple(frames.shape)}, {tuple(masks.shape)}")
        if k == 0:
            return self
        if self.n + k > MEAN_ACCUM_MAX_FRAMES:
            raise _lib.VuError(f"the masked-mean accumulator holds at most {MEAN_ACCUM_MAX_FRAMES} frames: {self.n} + {k}")
        rc = _lib.ERR_UNSUPPORTED
        if (self.ksize, self.iters) == (3, 2):
            rc = lib().vu_masked_mean_accum_add_dilate32(_p(self.state), _p(frames), _p(masks), k, self.h, self.w, _stream())
        if rc == _lib.ERR_UNSUPPORTED:
            d = dilate(masks, self.ksize, self.iters)
            rc = lib().vu_masked_mean_accum_add(_p(self.state), _p(frames), _p(d), k, self.h * self.w, _stream())
        check(rc)
        self.n += k
        return self

    def result(self):
        if self.n < 1:
            raise _lib.VuError("the masked-mean accumulator holds no frames")
        bg = torch.empty((self.h, self.w, 3), dtype=u8, device=self.device)
        always = torch.empty((self.h, self.w), dtype=u8, device=self.device)
        check(lib().vu_masked_mean_accum_finish(_p(self.state), self.h * self.w, self.min_count, _p(bg), _p(always), _stream()))
        return bg, always


# ---- per-frame branches on the device (batched clips) --------------------------------

def cf_samples(hsv_lo, mask_lo, mask_op, max_samples, prior=None, invert=False):
    """training samples of the mixtures gathered on the device (colorfiltering/agent.py:139-141): every
    (len // max_samples)-th selected pixel in row-major order.  selection = (mask < 128 if mask_op == 0 else mask > 128)
    and, with ``prior`` = (lo, hi), lo < H < hi (or its negation with ``invert``).  Returns (samples [3, n] uint8 numpy,
    number of selected pixels, histogram [256] of the H samples)."""
    hsv_lo, mask_lo = _img(hsv_lo), _mask(mask_lo)
    h, w = mask_lo.shape[-2:]
    cap = 2 * int(max_samples)
    samples = torch.empty((3, cap), dtype=u8, device=hsv_lo.device)
    meta = torch.empty(3, dtype=torch.int32, device=hsv_lo.device)
    hist = torch.empty(256, dtype=torch.int32, device=hsv_lo.device)
    ws_bytes = int(lib().vu_cf_samples_workspace_bytes(h))
    ws = torch.empty(ws_bytes, dtype=u8, device=hsv_lo.device)
    mode = 0 if prior is None else (2 if invert else 1)
    lo, hi = (0, 0) if prior is None else (int(prior[0]), int(prior[1]))
    check(lib().vu_cf_samples(_p(hsv_lo), _p(mask_lo), h, w, int(mask_op), mode, lo, hi, int(max_samples), _p(samples), cap, _p(meta), _p(hist),
                              _p(ws), ws_bytes, _stream()))
    total, _, kept = (int(v) for v in meta.cpu())
    return samples[:, :kept].cpu().numpy(), total, hist.cpu().numpy()


def ratio_flags(counts2, thr):
    counts2 = _dev(counts2, torch.int64)
    n = counts2.shape[0]
    flags = torch.empty(n, dtype=u8, device=counts2.device)
    check(lib().vu_ratio_flags(_p(counts2), n, float(thr), _p(flags), _stream()))
    return flags


def count_gt_lt(x, thr, item_ndim=2):
    """[n,2] int64: (#{x > thr}, #{x < thr}) per item, one pass."""
    x = _dev(x)
    n, per = _items(x, item_ndim)
    out = torch.empty((n, 2), dtype=torch.int64, device=x.device)
    check(lib().vu_count_gt_lt_u8(_p(x), n, per, int(thr), _p(out), _stream()))
    return out


def cf_degenerate_flags(masks, fg_min, bg_min):
    """per-frame early-out flags of ColorFilteringAgent.forward from the segmentation masks"""
    c = count_gt_lt(masks, 128)
    n = c.shape[0]
    flags = torch.empty(n, dtype=u8, device=c.device)
    second = ctypes.c_void_p(c.data_ptr() + 8)
    check(lib().vu_cf_degenerate_flags(_p(c), second, n, 2, int(fg_min), int(bg_min), _p(flags), _stream()))
    return flags


def select_frames(a, b, flags):
    """out[i] = a[i] if flags[i] else b[i] (whole frames)."""
    a, b, flags = _dev(a), _dev(b), _dev(flags)
    n = a.shape[0]
    out = torch.empty_like(a)
    check(lib().vu_select_frames(_p(a), _p(b), _p(flags), n, a.numel() // n, _p(out), _stream()))
    return out


def set128_unflagged(a, b, flags):
    a, b, flags = _dev(a), _dev(b), _dev(flags)
    n = a.shape[0]
    out = torch.empty_like(a)
    check(lib().vu_set128_unflagged(_p(a), _p(b), _p(flags), n, a.numel() // n, _p(out), _stream()))
    return out


# ---- BackgroundAgent pieces (bgmodel/agent.py 'mean' / 'pcov') ------------------------------------

def mask_bbox(mask):
    """(min row, max row, min col, max col) of mask > 0 as python ints, or None for an empty mask (one host read-back)"""
    mask = _mask(mask)
    h, w = mask.shape
    out = torch.empty(4, dtype=torch.int32, device=mask.device)
    check(lib().vu_mask_bbox(_p(mask), h, w, _p(out), _stream()))
    r0, r1, c0, c1 = (int(v) for v in out.cpu())
    return None if r1 < 0 else (r0, r1, c0, c1)


def masked_sum3(img, mask=None):
    """-> (sums [3] python ints, count) of img [H,W,3] over mask > 0 (all pixels without a mask); one host read-back"""
    img = _img(img)
    out = torch.empty(4, dtype=torch.int64, device=img.device)
    check(lib().vu_masked_sum3(_p(img), _p(_mask(mask)) if mask is not None else None, img.numel() // 3, _p(out), _stream()))
    v = [int(x) for x in out.cpu()]
    return v[:3], v[3]


def pcov_fill(img, hole_mask, box, ksize=5, max_rounds=100, batch=8):
    """get_bg_by_pcov's loop (bgmodel/agent.py:118-129) on box = (x0, x1, y0, y1) (rows, columns) of img [H,W,3] with the
    hole = hole_mask > 0.  Returns the filled box [x1-x0, y1-y0, 3].  Rounds are enqueued ``batch`` at a time; finished
    rounds return at once on the device."""
    img, hole_mask = _img(img), _mask(hole_mask)
    h, w = hole_mask.shape
    x0, x1, y0, y1 = box
    rh, rw = x1 - x0, y1 - y0
    dev = img.device
    bufs = [torch.empty((rh, rw, 3), dtype=u8, device=dev) for _ in range(2)]
    valid = [torch.empty((rh, rw), dtype=u8, device=dev) for _ in range(2)]
    flags = torch.zeros(max_rounds + 1, dtype=torch.int32, device=dev)
    off = x0 * w + y0
    done_after = max_rounds
    r = 0
    while r < max_rounds:
        for _ in range(min(batch, max_rounds - r)):
            if r == 0:
                src_i, src_v, pitch = ctypes.c_void_p(img.data_ptr() + 3 * off), ctypes.c_void_p(hole_mask.data_ptr() + off), w
            else:
                src_i, src_v, pitch = _p(bufs[r % 2]), _p(valid[r % 2]), rw
            check(lib().vu_pcov_round(src_i, src_v, pitch, int(r == 0), rh, rw, int(ksize), _p(bufs[(r + 1) % 2]), _p(valid[(r + 1) % 2]),
                                      _p(flags), r, _stream()))
            r += 1
        f = flags[1:r + 1].cpu().numpy()
        zero = np.flatnonzero(f == 0)
        if len(zero):                       # flags[k + 1] == 0: round k left no invalid pixel -> k + 1 rounds ran
            done_after = int(zero[0]) + 1
            break
    return bufs[done_after % 2]


# ---- regionfill (utils/region_fill.py) -----------------------------------------------------------------

def resize_linear_f64(x, dh, dw, fx=None, fy=None, keep_mask=None, keep_src=None):
    """cv2.resize of float64 planes [C,H,W] (default INTER_LINEAR).  fx / fy: the ``(0, 0), fx=, fy=`` form (sampling step
    1 / fx whatever the rounded size).  keep_mask / keep_src: where keep_mask == 0 the result is keep_src."""
    x = _dev(x, torch.float64)
    c, sh, sw = x.shape
    out = torch.empty((c, dh, dw), dtype=torch.float64, device=x.device)
    sx = 1.0 / fx if fx is not None else 1.0 / (float(dw) / sw)
    sy = 1.0 / fy if fy is not None else 1.0 / (float(dh) / sh)
    if keep_mask is not None:
        keep_mask, keep_src = _mask(keep_mask), _dev(keep_src, torch.float64)
        if tuple(keep_mask.shape) != (dh, dw) or tuple(keep_src.shape) != (c, dh, dw):
            raise ValueError("keep_mask / keep_src must have the output's shape")
    check(lib().vu_resize_linear_f64(_p(x), c, sh, sw, _p(out), int(dh), int(dw), sx, sy,
                                     _p(keep_mask) if keep_mask is not None else None, _p(keep_src) if keep_src is not None else None, _stream()))
    return out


def laplace_fill(planes, mask, tol=1e-10, max_iters=None, snap_eps=1e-6):
    """regionfillLaplace (utils/region_fill.py:26-63) for float64 planes [C,H,W] sharing mask [H,W] (> 0 = fill): solved on
    the mask's bounding box (+ 1 pixel, so that only real image borders act as borders).  -> (filled planes, iterations).
    Filled values within ``snap_eps`` of an integer are set to it (the callers truncate to uint8; include/vu_b200.h).
    Raises if the conjugate gradients did not reach ``tol`` (relative residual) within ``max_iters``, by default the
    number of pixels in that box (at least 50000): in exact arithmetic CG ends within as many iterations as there are
    unknowns, so a valid mask of any size gets a cap it cannot need."""
    planes, mask = _dev(planes, torch.float64), _mask(mask)
    c, h, w = planes.shape
    if tuple(mask.shape) != (h, w):
        raise ValueError("mask must be [H,W] of the planes")
    box = mask_bbox(mask)
    out = planes.clone()
    if box is None:
        return out, 0
    r0, r1, c0, c1 = box
    r0, r1, c0, c1 = max(r0 - 1, 0), min(r1 + 2, h), max(c0 - 1, 0), min(c1 + 2, w)
    x = out[:, r0:r1, c0:c1].contiguous()
    m = mask[r0:r1, c0:c1].contiguous()
    rh, rw = r1 - r0, c1 - c0
    if max_iters is None:
        max_iters = max(50000, rh * rw)
    nbytes = lib().vu_regionfill_workspace_bytes(c, rh, rw)
    ws = torch.empty(nbytes, dtype=u8, device=planes.device)
    iters, resid = ctypes.c_int32(0), ctypes.c_double(0.0)
    check(lib().vu_regionfill_f64(_p(x), _p(m), c, rh, rw, float(tol), int(max_iters), float(snap_eps), _p(ws), nbytes, ctypes.byref(iters), ctypes.byref(resid), _stream()))
    if not resid.value <= tol:
        raise RuntimeError(f"regionfill: residual {resid.value:.3g} after {iters.value} iterations (tol {tol:g})")
    out[:, r0:r1, c0:c1] = x
    return out, iters.value


def regionfill(planes, mask, factor=1.0, tol=1e-10):
    """regionfill (utils/region_fill.py:7-17) for planes [C,H,W] (any real dtype; uint8 images as they are) sharing mask
    [H,W] (bool / uint8, != 0 = fill).  -> float64 [C,H,W]."""
    mask = _mask(mask)
    if not (isinstance(planes, torch.Tensor) and planes.is_cuda and planes.ndim == 3):
        raise TypeError("expected a CUDA tensor [C,H,W]")
    src = planes.to(torch.float64).contiguous()
    c, h, w = src.shape
    if factor == 1.0:
        return laplace_fill(src, mask, tol)[0]
    dw, dh = int(np.rint(w * factor)), int(np.rint(h * factor))          # saturate_cast<int>: round half to even
    m_lo = (resize_linear_f64(mask[None].to(torch.float64), dh, dw, factor, factor)[0] > 0).to(u8)
    x_lo = resize_linear_f64(src, dh, dw, factor, factor)
    x_lo = laplace_fill(x_lo, m_lo, tol)[0]
    return resize_linear_f64(x_lo, h, w, keep_mask=mask, keep_src=src)


# ---- remove_invalid_objects (utils/maskprocess.py:77-152) -----------------------------------------

def remove_invalid_objects(alpha, segmask, score_map, saliency_thr, consensus_thr, max_objects=16384, out=None):
    """alpha / segmask [H,W] or [N,H,W]; score_map [H,W] float64 device tensor.  -> (out, status): status [n] int32 device
    tensor = contours per frame, > max_objects where a frame overflowed (output undefined there; the caller checks)."""
    alpha, segmask = _mask(alpha), _mask(segmask)
    if segmask.shape != alpha.shape:
        raise ValueError("segmask must have alpha's shape")
    score_map = _dev(score_map, torch.float64)
    h, w = alpha.shape[-2:]
    if tuple(score_map.shape) != (h, w):
        raise ValueError("score_map must be [H,W]")
    n = 1 if alpha.ndim == 2 else alpha.shape[0]
    out = _out(out, alpha.shape, alpha.device)
    status = torch.empty(n, dtype=torch.int32, device=alpha.device)
    ws_bytes = int(lib().vu_remove_objects_workspace_bytes(n, h, w, int(max_objects)))
    ws = torch.empty(ws_bytes, dtype=u8, device=alpha.device)
    check(lib().vu_remove_invalid_objects(_p(alpha), _p(segmask), _p(score_map), n, h, w, float(saliency_thr), float(consensus_thr), _p(out),
                                          _p(status), _p(ws), ws_bytes, int(max_objects), _stream()))
    return out, status


# ---- frame I/O glue (utils/fileio.py) ----------------------------------------------------------------

def planar_rgb_to_bgr(x):
    """[3,H,W] planar RGB (what nvJPEG decodes to) -> [H,W,3] interleaved BGR"""
    x = _dev(x)
    h, w = x.shape[-2:]
    out = torch.empty((h, w, 3), dtype=u8, device=x.device)
    check(lib().vu_planar_rgb_to_bgr(_p(x), _p(out), h * w, _stream()))
    return out


def bgr_to_planar_rgb(x):
    """[H,W,3] interleaved BGR -> [3,H,W] planar RGB (what nvJPEG encodes from)"""
    x = _img(x)
    h, w = x.shape[:2]
    out = torch.empty((3, h, w), dtype=u8, device=x.device)
    check(lib().vu_bgr_to_planar_rgb(_p(x), _p(out), h * w, _stream()))
    return out
