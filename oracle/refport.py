"""Restatement of the reference's hot-path functions on top of ``cvmodel``.

TEST INFRASTRUCTURE (see ``oracle/__init__.py``).  Every function cites the
reference lines it follows (paths relative to the reference root).  Arrays are
numpy uint8, HWC, BGR, masks HW -- the reference's conventions.  Nothing here
mutates its arguments.
"""
import numpy as np

from . import cvmodel as cvm

# --------------------------------------------------------------------------
# size math / morphology wrappers
# --------------------------------------------------------------------------


def get_target_size(h, w, target_long_side, division=1):
    """unscreen/utils/imgprocess.py:164-192."""
    if h > w:
        th = target_long_side
        tw = int(float(target_long_side) * w / h)
        if tw % division != 0:
            tw = (tw // division + 1) * division
    else:
        tw = target_long_side
        th = int(float(target_long_side) * h / w)
        if th % division != 0:
            th = (th // division + 1) * division
    return th, tw


def adaptive_resize(img, img_target):
    """unscreen/utils/imgprocess.py:33-37."""
    return cvm.resize_linear(img, img_target.shape[1], img_target.shape[0])


def dilate_mask(mask, kernelsize=5, iters=10):
    """unscreen/utils/maskprocess.py:7-19."""
    return cvm.dilate(mask, kernelsize, iters)


def erode_mask(mask, kernelsize=5, iters=10):
    """unscreen/utils/maskprocess.py:22-34."""
    return cvm.erode(mask, kernelsize, iters)


def exist_foreground(mask, fg_exist_thr):
    """unscreen/utils/maskprocess.py:56-60 (strict '>')."""
    h, w = mask.shape
    return bool(int((mask >= 128).sum()) > fg_exist_thr * h * w)


def get_outer_boundary(mask, kernelsize=7, iters=10):
    """unscreen/utils/maskprocess.py:63-74: uint8 subtraction wraps, the clip
    is a no-op."""
    d = dilate_mask(mask, kernelsize, iters)
    return (d - mask).astype(np.uint8)


# --------------------------------------------------------------------------
# is_pixel_inrange
# --------------------------------------------------------------------------


def is_pixel_inrange(img, bgimg, winsize=(20, 20, 120), long_side_input=-1):
    """unscreen/utils/fgfuncs.py:9-65.  ``bgimg`` is (h,w,3) or (3,)."""
    assert bgimg.ndim == 3 or bgimg.ndim == 1
    h, w = img.shape[:2]
    if long_side_input > 0:
        ih, iw = get_target_size(h, w, long_side_input)
        img = cvm.resize_linear(img, iw, ih)
        if bgimg.ndim == 3:
            bgimg = cvm.resize_linear(bgimg, iw, ih)
    hsv = cvm.bgr2hsv(img).astype(np.int32)
    half = np.array(winsize, dtype=np.int32) // 2
    if bgimg.ndim == 3:
        bg = cvm.bgr2hsv(bgimg).astype(np.int32)
    else:
        bg = cvm.bgr2hsv(bgimg[None, None, :])[0, 0].astype(np.int32)
    lo = np.clip(bg - half, 10, 255)
    hi = np.clip(bg + half, 10, 255)
    mask = np.all((hsv >= lo) & (hsv <= hi), axis=-1)
    if long_side_input > 0:
        # fgfuncs.py:51,63: INTER_NEAREST lands in the dst slot => bilinear
        m8 = mask.astype(np.uint8) * (1 if bgimg.ndim == 3 else 255)
        mask = cvm.resize_linear(m8, w, h) > 0
    return mask


# --------------------------------------------------------------------------
# colour filtering
# --------------------------------------------------------------------------

POW_EXP = np.float64(np.float32(1 / 3.))  # torch casts the python double to f32


def gmm_lut(means, covariances, weights):
    """256-entry float32 table of ColorFilteringAgent.get_prob_by_gmm
    (unscreen/colorfiltering/agent.py:201-230) evaluated on samples 0..255.
    Uses the same torch CPU ops in the same order as the reference, so the
    table is bitwise what the reference computes per pixel (SURVEY.md A.6)."""
    import torch
    means = np.asarray(means, dtype=np.float64).reshape(-1)
    stds = np.sqrt(np.asarray(covariances, dtype=np.float64).reshape(-1))
    weights = np.asarray(weights, dtype=np.float64).reshape(-1)
    samples = np.arange(256, dtype=np.float64).reshape(1, -1)
    samples_t = torch.from_numpy(samples).float()
    means_t = torch.from_numpy(means[..., np.newaxis]).float()
    stds_t = torch.from_numpy(stds[..., np.newaxis]).float()
    weights_t = torch.from_numpy(weights).float().unsqueeze(dim=0)
    x = (samples_t - means_t) / stds_t
    y = 1. / (stds_t * np.sqrt(2 * np.pi)) * torch.exp(-1. / 2 * torch.pow(x, 2))
    prob = torch.mm(weights_t, y).squeeze()
    return prob.numpy().astype(np.float32).reshape(256)


def gmm_luts_from_models(gmms):
    """three sklearn GaussianMixture (spherical) -> (3,256) float32."""
    return np.stack([gmm_lut(g.means_.squeeze(), g.covariances_.squeeze(), g.weights_.squeeze())
                     for g in gmms])


def pow_third(x):
    """torch.pow(x_f32, 1/3.) model: the exponent is the *float32* nearest to
    1/3 (0.3333333432674408); evaluated in float64 and rounded once to
    float32.  torch's SLEEF powf is a 1-ULP routine, so 1.8 % of values differ
    from this by one ULP on this container's AVX-512 build -- irreproducible
    across CPUs, and invisible after the uint8 cast except within ~1e-5 of an
    integer boundary."""
    x = np.asarray(x, dtype=np.float32).astype(np.float64)
    with np.errstate(all="ignore"):
        return np.power(x, POW_EXP).astype(np.float32)


def alpha_from_luts(img_hsv, lut_bg, lut_fg):
    """ColorFilteringAgent.get_alpha_by_gmm, unscreen/colorfiltering/agent.py:
    232-257, with the per-channel mixtures folded into tables."""
    f = np.float32
    h = img_hsv[..., 0]
    s = img_hsv[..., 1]
    v = img_hsv[..., 2]
    bg = ((f(1.0) * lut_bg[0][h]).astype(f) * lut_bg[1][s]).astype(f) * lut_bg[2][v]
    fg = ((f(1.0) * lut_fg[0][h]).astype(f) * lut_fg[1][s]).astype(f) * lut_fg[2][v]
    bg = pow_third(bg.astype(f))
    fg = pow_third(fg.astype(f))
    den = ((bg + fg).astype(f) + f(1e-6)).astype(f)
    prob = (fg / den).astype(f)
    return np.clip((prob * f(255)).astype(f), 0, 255).astype(np.uint8)


def cf_postprocess(alpha, mask, thr_ratio=0.8):
    """ColorFilteringAgent.postprocess, unscreen/colorfiltering/agent.py:
    259-283.  Empty consistent area => NaN threshold => nothing zeroed."""
    alpha = alpha.copy()
    sel = (alpha > 128) & (mask > 0)
    n = int(sel.sum())
    if n > 0:
        thr = alpha[sel].astype(np.float64).mean() * thr_ratio
        alpha[alpha < thr] = 0
    alpha = erode_mask(dilate_mask(alpha, 3, 2), 3, 2)
    alpha = dilate_mask(erode_mask(alpha, 3, 2), 3, 2)
    return alpha


def get_color_prior(img_hsv, mask, winsize, max_num_samples=10000):
    """ColorFilteringAgent.get_color_prior, agent.py:113-146.  Returns
    (mask_by_prior, peak)."""
    samples = img_hsv[:, :, 0][mask]
    if len(samples) > max_num_samples:
        samples = samples[::len(samples) // max_num_samples]
    hist = np.bincount(samples.astype(np.int64), minlength=256)[:256]
    peak = int(np.argmax(hist))
    hch = img_hsv[:, :, 0].astype(np.int64)
    return (hch > peak - winsize // 2) & (hch < peak + winsize // 2), peak


def strided_samples(channel, mask, max_num_samples=10000):
    """the ordered, strided sample gather of agent.py:163-167 / 190-194."""
    s = channel[mask].astype(np.float64)
    if len(s) > max_num_samples:
        s = s[::len(s) // max_num_samples]
    return s


def bg_color_hsv(bg_means0):
    """agent.py:345-351: int(mean(component-0 mean)) per channel."""
    return np.array([int(np.mean(m)) for m in bg_means0], dtype=np.uint8)


def cf_forward_predict(img, mask, lut_bg, lut_fg, bg_hsv, input_long_side=960,
                       fg_ncomp=(10, 10, 10), bg_ncomp=(3, 5, 5)):
    """ColorFilteringAgent.forward(img, mask, iters=0), agent.py:285-354, with
    the fitted mixtures supplied as tables + the component-0 mean colour."""
    if int((mask > 128).sum()) < max(fg_ncomp) * 5:
        return mask, img, 1.0
    if int((mask < 128).sum()) < max(bg_ncomp) * 5:
        return mask, np.zeros_like(img), 1.0
    hsv = cvm.bgr2hsv(img)
    oh, ow = hsv.shape[:2]
    th, tw = get_target_size(oh, ow, input_long_side)
    hsv_lo = cvm.resize_linear(hsv, tw, th)
    mask_lo = cvm.resize_linear(mask, tw, th)
    alpha = alpha_from_luts(hsv_lo, lut_bg, lut_fg)
    alpha = cf_postprocess(alpha, mask_lo)
    alpha = cvm.resize_linear(alpha, ow, oh)
    bg_img = cvm.hsv2bgr(np.broadcast_to(np.asarray(bg_hsv, np.uint8), (oh, ow, 3)))
    return alpha, bg_img, None


# --------------------------------------------------------------------------
# trimap
# --------------------------------------------------------------------------


def generate_trimap(mask, input_long_side=960, kernelsize=3, iters=5):
    """TrimapAgent.generate_trimap, unscreen/trimap/agent.py:35-61.  The
    up-scale at :59 is bilinear (INTER_NEAREST is passed in the dst slot)."""
    oh, ow = mask.shape
    ih, iw = get_target_size(oh, ow, input_long_side)
    m = cvm.resize_nearest(mask, iw, ih)
    tri = np.full((ih, iw), 128, np.uint8)
    dil = dilate_mask(m, kernelsize, iters)
    ero = erode_mask(m, kernelsize, iters)
    tri[ero > 127] = 255
    tri[dil < 128] = 0
    tri = cvm.resize_linear(tri, ow, oh)
    tri[(tri > 0) & (tri < 255)] = 128
    return tri


def generate_trimap_withbg(mask, img, bgimg, input_long_side=960, kernelsize=3, iters=5,
                           color_winsize=(10, 100, 180)):
    """TrimapAgent.generate_trimap_withbg, unscreen/trimap/agent.py:63-101."""
    npos = int((mask > 0).sum())
    if npos == 0:
        return mask
    bgmask = is_pixel_inrange(img, bgimg, color_winsize)
    fuzzy = (mask > 0) & bgmask
    if float(fuzzy.sum()) / npos > 0.1:
        return generate_trimap(mask, input_long_side, kernelsize, iters)
    ens = mask.copy()
    ens[fuzzy] = 0
    tri = generate_trimap(ens, input_long_side, kernelsize, iters)
    tri[fuzzy] = 128
    return tri


# --------------------------------------------------------------------------
# compositing family
# --------------------------------------------------------------------------


def fg_hsv_stage(img, alpha, bg):
    """the exactly reproducible part of get_fg (fgfuncs.py:100-108): float32
    HSV arithmetic, clamp, truncate -- before the +-1 HSV2BGR."""
    f = np.float32
    ih = cvm.bgr2hsv(img).astype(f)
    bh = cvm.bgr2hsv(bg).astype(f)
    a = (alpha.astype(f) / f(255.))[..., None]
    t = ((f(1) - a).astype(f) * bh).astype(f)
    fg = np.clip((ih - t).astype(f), 0, 255)
    return fg.astype(np.uint8)


def get_fg(img, alpha, bg):
    """unscreen/utils/fgfuncs.py:84-110."""
    return cvm.hsv2bgr(fg_hsv_stage(img, alpha, bg))


def bg_hsv_stage(alpha, bg):
    f = np.float32
    bh = cvm.bgr2hsv(bg).astype(f)
    a = (alpha.astype(f) / f(255.))[..., None]
    out = np.clip(((f(1) - a).astype(f) * bh).astype(f), 0, 255)
    return out.astype(np.uint8)


def get_bg(alpha, bg):
    """unscreen/utils/fgfuncs.py:113-137."""
    return cvm.hsv2bgr(bg_hsv_stage(alpha, bg))


def get_fg_naive(img, alpha):
    """unscreen/utils/fgfuncs.py:68-81 (float64)."""
    a = alpha.astype(np.float64) / 255.
    return (img.astype(np.float64) * a[..., None]).astype(np.uint8)


def fuse_fgbg(fg, bg, mask):
    """unscreen/utils/visualize.py:7-24 (float64)."""
    a = mask.astype(np.float64)[..., None] / 255
    return (a * fg.astype(np.float64) + (1 - a) * bg.astype(np.float64)).astype(np.uint8)


def composite_fgbg(fg, alpha, bg, extend=False):
    """unscreen/utils/fgfuncs.py:172-214."""
    fg_h, fg_w = fg.shape[:2]
    bg_h, bg_w = bg.shape[:2]
    if float(fg_h) / fg_w > float(bg_h) / bg_w:
        nh = fg_h
        nw = int(float(bg_w) * nh / bg_h)
    else:
        nw = fg_w
        nh = int(float(bg_h) * nw / bg_w)
    bg = cvm.resize_linear(bg, nw, nh)
    left = max(nw // 2 - fg_w // 2, 0)
    top = max(nh // 2 - fg_h // 2, 0)
    a = alpha.astype(np.float64) / 255.
    a[a > 0.9] = 1
    roi = bg[top:top + fg_h, left:left + fg_w].astype(np.float64)
    comp = (fg.astype(np.float64) + roi * (1 - a[..., None])).clip(0, 255).astype(np.uint8)
    if extend:
        out = bg.copy()
        out[top:top + fg_h, left:left + fg_w] = comp
        return out
    return comp


def replace_blend(fg, mask3, bg):
    """tools/replace/replace.py:74-76 (float64; mask has the image's shape, or
    HW for the single-channel variant of BASELINE config 4)."""
    m = mask3.astype(np.float64) / 255
    if m.ndim == 2:
        m = m[..., None]
    res = fg.astype(np.float64) * m + bg.astype(np.float64) * (1 - m)
    return res.astype(np.uint8)


def shift_fg(img, dx=0, dy=0):
    """unscreen/utils/imgprocess.py:55-64."""
    return cvm.warp_translate(img, dx, dy)


def rescale_fg(img, scale_factor=1.1):
    """unscreen/utils/imgprocess.py:40-52 (see the parity note of
    ``cvmodel.resize_cubic_crop``)."""
    return cvm.resize_cubic_crop(img, scale_factor)


def replace_frame(fg, mask, bg, dx, dy, scale_factor=1.2):
    """tools/replace/replace.py:69-76: shift and rescale the foreground and its
    mask, then blend over the (already resized) new background."""
    fg_s = rescale_fg(shift_fg(fg, dx, dy), scale_factor)
    mk_s = rescale_fg(shift_fg(mask, dx, dy), scale_factor)
    return replace_blend(fg_s, mk_s, bg)


def nearest_index(dst, src):
    """source indices of torch.nn.functional.interpolate(mode='nearest') on the
    CPU for one axis: identity for equal sizes, i >> 1 for an exact doubling,
    else floor(float32(i) * float32(src / dst)) clamped."""
    i = np.arange(dst)
    if dst == src:
        return i
    if dst == 2 * src:
        return i >> 1
    scale = np.float32(src) / np.float32(dst)
    return np.minimum(np.floor(i.astype(np.float32) * scale).astype(np.int64), src - 1)


COLOR_CORRECT_MAX_ITERS = 24


def color_correct(img, alpha, bg_color, target_long_side=960, mean_exp=0.95):
    """unscreen/utils/imgprocess.py:263-300: chroma distance to the background
    colour in Lab at the working resolution, normalised, square-rooted until
    its mean over the matte reaches ``mean_exp``, and multiplied into alpha.

    float32 like the reference (torch CPU) except for one thing: the mean of
    the loop condition is accumulated in float64 here (torch sums float32 in an
    implementation-defined order), so the iteration count can differ only when
    the reference's mean lies within float32 summation noise of ``mean_exp``."""
    f32 = np.float32
    h, w = img.shape[:2]
    th, tw = get_target_size(h, w, target_long_side)
    lab = cvm.bgr2lab(cvm.resize_linear(img, tw, th))
    bg = cvm.bgr2lab(np.asarray(bg_color, np.uint8).reshape(1, 1, 3))
    d = (lab.astype(f32) / f32(255.0))[:, :, 1:] - (bg.astype(f32) / f32(255.0))[:, :, 1:]
    dist = np.sqrt(d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1])
    lo, hi = dist.min(), dist.max()
    with np.errstate(invalid="ignore", divide="ignore"):
        dist = ((dist - lo) / (hi - lo)).astype(f32)
    a_lo = cvm.resize_linear(alpha, tw, th)
    sel = (a_lo > 0) & (dist > 0)
    for _ in range(COLOR_CORRECT_MAX_ITERS):
        if not sel.any() or not (dist[sel].mean(dtype=np.float64) < mean_exp):
            break
        dist = np.sqrt(dist)
    dist[a_lo == 0] = 0
    dist = dist[nearest_index(h, th)][:, nearest_index(w, tw)]
    with np.errstate(invalid="ignore"):
        out = alpha.astype(f32) * dist
    return np.where(np.isnan(out), 0, out).astype(np.uint8)


def patch_bg(bgimg, frame, alpha, mode):
    """tools/unscreen/green.py:125 (mode 'lt128') and bg.py:99 /
    bg_offline.py:171 (mode 'eq0'): predicated copy frame -> bgimg."""
    out = bgimg.copy()
    sel = (alpha < 128) if mode == "lt128" else (alpha == 0)
    out[sel] = frame[sel]
    return out


def fuse_bg(bgimg, bg_always, beta):
    """tools/unscreen/bg_offline.py:150-151: float32 array math with python
    float scalars (scalars round to float32)."""
    f = np.float32
    return ((bgimg.astype(f) * f(beta)).astype(f) + (f(1 - beta) * bg_always.astype(f)).astype(f)).astype(np.uint8)


def bgdiff_gate(frame, bgimg, mask, thr=25):
    """tools/unscreen/bg.py:85-92 == bg_offline.py:154-160: absdiff ->
    BGR2GRAY -> '>thr -> 255' (values <=thr are kept) -> dilate(4,2) ->
    mask * (g // 255)."""
    raw = np.abs(frame.astype(np.int32) - bgimg.astype(np.int32)).astype(np.uint8)
    g = cvm.bgr2gray(raw)
    g = g.copy()
    g[g > thr] = 255
    g = dilate_mask(g, 4, 2)
    return (mask * (g // 255)).astype(np.uint8)


def binarise_dilate(alpha):
    """tools/unscreen/bg.py:74-77."""
    a = np.where(alpha > 128, 255, 0).astype(np.uint8)
    return dilate_mask(a, 3, 2)


# --------------------------------------------------------------------------
# temporal reducers
# --------------------------------------------------------------------------


def masked_temporal_mean(frames, masks, ksize=3, iters=2, min_count=10):
    """tools/unscreen/bg_offline.py:106-125 (dead code in the reference; the
    only temporal background estimator it contains).  ``masks`` is [N,H,W]
    (single channel; the reference's 3-identical-channel JPEG masks give the
    same result per channel).  Returns (bg_always HxWx3 u8, mask_always HxW u8).
    The TELEA inpaint at :127-129 is out of scope."""
    n, h, w, _ = frames.shape
    acc = np.zeros((h, w, 3), np.int64)
    cnt = np.zeros((h, w), np.int64)
    for i in range(n):
        m = dilate_mask(masks[i], ksize, iters)
        keep = (1 - (m // 255).astype(np.int64))
        acc += frames[i].astype(np.int64) * keep[..., None]
        cnt += (m < 250)
    mask_always = ((cnt <= min_count) * 255).astype(np.uint8)
    den = np.maximum(cnt, 1).astype(np.float64)
    bg = np.clip(acc.astype(np.float64) / den[..., None], 0, 255).astype(np.uint8)
    bg[mask_always == 255] = 0
    return bg, mask_always


def temporal_median(frames):
    """NEW SPECIFICATION (SURVEY.md section 8 a23; the reference has no
    median): np.median(stack, 0).astype(np.uint8); for even N this equals
    (sorted[N/2-1] + sorted[N/2]) >> 1."""
    n = frames.shape[0]
    k = (n - 1) // 2
    part = np.partition(frames, (k, n // 2), axis=0)
    lo = part[k].astype(np.uint16)
    hi = part[n // 2].astype(np.uint16)
    return ((lo + hi) >> 1).astype(np.uint8)


# --------------------------------------------------------------------------
# BackgroundAgent (SURVEY 8f rank 4): 'mean' and 'pcov' branches; 'rf' (sparse
# Laplace solve with scipy) is not restated
# --------------------------------------------------------------------------

def get_fgbox(fgmask, padsize=5):
    """unscreen/utils/maskprocess.py:37-53 (rows first: 'left/right' are row bounds, 'top/bottom' column bounds)."""
    h, w = fgmask.shape
    x, y = np.where(fgmask > 0)
    left, right, top, bottom = np.min(x), np.max(x), np.min(y), np.max(y)
    return max(left - padsize, 0), min(right + padsize, h), max(top - padsize, 0), min(bottom + padsize, w)


def box_sum(a, k):
    """k x k window sums with cv2's default BORDER_REFLECT_101; a is [H,W] or [H,W,C] int64.  A window reaches k//2
    up / left and k - 1 - k//2 down / right of its anchor (cv2's default anchor: the window centre)."""
    r0, r1 = k // 2, k - 1 - k // 2
    pad = ((r0, r1), (r0, r1)) + ((0, 0),) * (a.ndim - 2)
    p = np.pad(a, pad, mode="reflect")
    h, w = a.shape[:2]
    s = np.zeros(a.shape, np.int64)
    for dy in range(k):
        for dx in range(k):
            s += p[dy:dy + h, dx:dx + w]
    return s


def box_filter_u8(img, k):
    """cv2.boxFilter(uint8, -1, (k,k)): the rounded window mean (k*k odd: the mean is never a tie)"""
    s = box_sum(img.astype(np.int64), k)
    return ((2 * s + k * k) // (2 * k * k)).astype(np.uint8)


def bg_mean_hsv(img_hsv, mask, boundary_ksize=7, boundary_iters=10):
    """BackgroundAgent.get_mean_bg, unscreen/bgmodel/agent.py:66-93 -> the HSV colour (3 uint8)."""
    boundary = get_outer_boundary(mask, boundary_ksize, boundary_iters) > 0
    n = int(boundary.sum())
    if n == 0:
        col = np.mean(img_hsv, axis=(0, 1))                  # float64, truncated by the uint8 assignment of :91
    else:
        col = (img_hsv * boundary[..., None]).sum(axis=(0, 1)) / n
    return col.astype(np.uint8)


def bg_by_pcov(img, mask, ksize=5):
    """BackgroundAgent.get_bg_by_pcov, unscreen/bgmodel/agent.py:95-131: iterated normalised box filters of the image
    with the hole zeroed and of the 0/1 validity map; pixels whose window saw a valid pixel take mean / validity
    (float64 division, clipped, truncated by the uint8 store) and become valid; stops once every pixel of the box
    around the hole is valid, after at most 100 rounds.  EVERY round re-filters the whole box, valid pixels too."""
    bgimg = img.copy()
    bgimg[mask > 0] = 0
    count = (mask == 0).astype(np.float64)
    x0, x1, y0, y1 = get_fgbox(mask, padsize=ksize)
    num_pixels = (x1 - x0) * (y1 - y0)
    count = count[x0:x1, y0:y1]
    roi = bgimg[x0:x1, y0:y1]
    for _ in range(100):
        roi = box_filter_u8(roi, ksize)
        count = box_sum(count.astype(np.int64), ksize).astype(np.float64) * (1.0 / (ksize * ksize))
        sel = count > 0
        roi[sel] = np.clip(roi[sel] / count[sel][..., None], 0, 255)      # float64 -> uint8 store truncates
        count[sel] = 1
        if count.sum() >= num_pixels:
            break
    bgimg[x0:x1, y0:y1] = roi
    return bgimg


def regionfill(I, mask, factor=1.0):
    """unscreen/utils/region_fill.py:7-63: fill the masked pixels of the single-channel image I with the solution of the
    discrete Laplace equation (every masked pixel = the mean of its in-image 4-neighbours; pixels outside the mask are
    the boundary data), at ``factor`` x the resolution, resized back and pasted under the mask.  -> float64 [H,W].
    The linear solve is scipy's ``spsolve``, like in the reference (scipy is the reference's dependency for this function);
    the two cv2.resize calls on float64 data are cvmodel.resize_linear_f64."""
    from scipy import sparse
    from scipy.sparse.linalg import spsolve
    I = np.asarray(I)
    mask = np.asarray(mask)
    if np.count_nonzero(mask) == 0:
        return I.copy()
    h0, w0 = I.shape
    if factor == 1.0:
        m, x = mask.astype(np.float64) > 0, I.astype(np.float64)
    else:
        dw, dh = cvm.scaled_size(w0, factor), cvm.scaled_size(h0, factor)
        m = cvm.resize_linear_f64(mask.astype(np.float64), dw, dh, factor, factor) > 0
        x = cvm.resize_linear_f64(I.astype(np.float64), dw, dh, factor, factor)
    h, w = m.shape
    ys, xs = np.nonzero(m)
    idx = -np.ones((h + 2, w + 2), np.int64)
    idx[ys + 1, xs + 1] = np.arange(ys.size)
    data = np.where(m, 0.0, x)                               # boundary data: every pixel outside the mask
    dpad = np.zeros((h + 2, w + 2))
    dpad[1:-1, 1:-1] = data
    nn = np.full((h, w), 4.0)
    nn[[0, -1], :] -= 1
    nn[:, [0, -1]] -= 1
    rows, cols, vals = [np.arange(ys.size)], [np.arange(ys.size)], [nn[ys, xs]]
    rhs = np.zeros(ys.size)
    for dy, dx in ((-1, 0), (0, 1), (1, 0), (0, -1)):
        nb = idx[ys + 1 + dy, xs + 1 + dx]
        k = nb >= 0
        rows.append(np.nonzero(k)[0])
        cols.append(nb[k])
        vals.append(-np.ones(int(k.sum())))
        rhs += dpad[ys + 1 + dy, xs + 1 + dx]
    D = sparse.coo_matrix((np.concatenate(vals), (np.concatenate(rows), np.concatenate(cols)))).tocsr()
    x = x.copy()
    x[ys, xs] = spsolve(D, rhs)
    out = x if (h, w) == (h0, w0) else cvm.resize_linear_f64(x, w0, h0)
    out = out.copy()
    keep = mask == 0
    out[keep] = I[keep]
    return out


def bg_by_regionfill(img_hsv, mask, boundary_ksize=7, boundary_iters=10):
    """BackgroundAgent.get_bg_by_regionfill, unscreen/bgmodel/agent.py:133-157: V from regionfill at half resolution,
    H and S from the boundary's mean colour."""
    col = bg_mean_hsv(img_hsv, mask, boundary_ksize, boundary_iters)
    out = img_hsv.copy()
    v = regionfill(img_hsv[:, :, 2], mask > 0, 0.5).astype(np.uint8)
    fgm = mask > 0
    out[fgm] = col
    out[:, :, 2][fgm] = v[fgm]
    return out


def background_forward(img, mask, method="rf", input_long_side=540, dilation_ksize=5, dilation_iters=3, boundary_ksize=7,
                       boundary_iters=10, pcov_ksize=5):
    """BackgroundAgent.forward, unscreen/bgmodel/agent.py:159-208."""
    oh, ow = mask.shape
    if (mask == 0).sum() == 0:
        return np.zeros(img.shape)                         # float64 zeros, as the reference returns them (:178)
    if mask.sum() == 0:
        return img
    ih, iw = get_target_size(oh, ow, input_long_side)
    img = cvm.resize_linear(img, iw, ih)
    mask = cvm.resize_linear(mask, iw, ih)
    dil = dilate_mask(mask, dilation_ksize, dilation_iters)
    if method == "mean":
        col = bg_mean_hsv(cvm.bgr2hsv(img), dil, boundary_ksize, boundary_iters)
        bg_hsv = np.empty(img.shape, np.uint8)
        bg_hsv[:] = col
        bgimg = fuse_fgbg(cvm.hsv2bgr(bg_hsv), img, dil)
    elif method == "pcov":
        bgimg = fuse_fgbg(bg_by_pcov(img, dil, pcov_ksize), img, dil)
    elif method == "rf":
        bgimg = cvm.hsv2bgr(bg_by_regionfill(cvm.bgr2hsv(img), dil, boundary_ksize, boundary_iters))
    else:
        raise NameError(f"No such method for background inpainting: {method}")
    return cvm.resize_linear(bgimg, ow, oh)


# --------------------------------------------------------------------------
# remove_invalid_objects (SURVEY 8f rank 2): closed-form model of
# cv2.findContours(RETR_LIST) + contourArea + drawContours(FILLED)
# --------------------------------------------------------------------------

def get_score_map(map_size, center):
    """unscreen/utils/maskprocess.py:155-178."""
    score_map = np.ones(map_size, np.float64)
    h, w = map_size
    y, x = int(h * center[0]), int(w * center[1])
    score_map[:, x:w] = np.linspace(0, 1, w - x)[np.newaxis, ...] ** 2
    score_map[:, 0:x] = np.linspace(1, 0, x)[np.newaxis, ...] ** 2
    score_map[y:h] += np.linspace(0, 1, h - y)[..., np.newaxis] ** 2
    score_map[0:y] += np.linspace(1, 0, y)[..., np.newaxis] ** 2
    score_map = np.sqrt(score_map)
    return (score_map.max() - score_map) / score_map.max()


def build_score_map(h, w, config):
    """unscreen/utils/maskprocess.py:181-189."""
    centers = config['objectremoval']['score_map_center']
    return get_score_map((h, w), centers['landscape'] if w > h else centers['portrait'])


def contour_objects(X):
    """Every contour cv2.findContours(X, RETR_LIST) returns, as (fill, area): ``fill`` = the pixels
    drawContours(.., FILLED) paints for it, ``area`` = cv2.contourArea of it.  X: bool [h,w].

    Foreground components are 8-connected, background components 4-connected, everything outside the image is one
    background component.  Two kinds of contour:
      * the outer border of a foreground component C.  Its polygon runs through C's border pixels; filled, it covers
        F = C and everything C encloses (holes, islands inside holes, ...).
      * the border of a hole H (a background component other than the outside), traced on the pixels of the surrounding
        component that are 4-adjacent to H (the ring).  Filled: H, the ring, and everything inside H.
    The polygon's vertices are pixel centres, so Pick's theorem gives its area from lattice-point counts, and the number
    B of chain steps of a border is a local count on the region it bounds: B = L - n1 for an outer border (L = pixel
    edges between F and its complement, n1 = 2x2 windows holding exactly one pixel of F) and B = L - n3 for a hole
    (edges between H' = H plus its inside and the ring; n3 = windows holding exactly three pixels of H').  Outer:
    area = |F| - B/2 - 1; hole: area = |H'| + B/2 - 1.  Checked against cv2 on thousands of random shapes
    (tests/test_oracle_vs_reference.py)."""
    from scipy import ndimage as ndi
    S8, S4 = np.ones((3, 3), int), np.array([[0, 1, 0], [1, 1, 1], [0, 1, 0]])
    P = np.pad(np.asarray(X, bool), 2)
    fl, nf = ndi.label(P, S8)
    bl, nb = ndi.label(~P, S4)

    def local(F):
        F = F.astype(np.int8)
        q = F[:-1, :-1] + F[:-1, 1:] + F[1:, :-1] + F[1:, 1:]
        L = int((F[:, :-1] != F[:, 1:]).sum() + (F[:-1, :] != F[1:, :]).sum())
        return L, int((q == 1).sum()), int((q == 3).sum())
    objs = []
    for c in range(1, nf + 1):
        comp = fl == c
        rest, _ = ndi.label(~comp, S4)
        fill = rest != rest[0, 0]
        L, n1, _ = local(fill)
        objs.append((fill[2:-2, 2:-2], fill.sum() - (L - n1) / 2.0 - 1))
    for b in range(1, nb + 1):
        if b == bl[0, 0]:
            continue
        hole = bl == b
        ys, xs = np.nonzero(hole)
        parent = fl[ys[0], xs[ys == ys[0]].min() - 1]     # the pixel left of the hole's first pixel (raster order)
        ring = (fl == parent) & ndi.binary_dilation(hole, S4)
        outside, _ = ndi.label(~hole, S8)
        inner = (outside != outside[0, 0]) & ~hole        # islands inside the hole
        hp = hole | inner
        L, _, n3 = local(hp)
        objs.append(((hp | ring)[2:-2, 2:-2], hp.sum() + (L - n3) / 2.0 - 1))
    return objs


def contour_records(X, segmask, score_map):
    """The closed form of ``contour_objects`` in whole-array operations: one labelling per class instead of one per
    contour (remove_invalid_objects_fast, one x86 core: 0.3 s for a blobby 1080p matte with 1 500 contours, 3.7 s for a
    4K noise matte with 350 000).  X: bool [h,w]; segmask uint8 [h,w]; score_map
    float64 [h,w].  Returns (records, lab, parent, nf):

      records: dict of per-contour arrays, one entry per contour (every label but the outside), in label order:
        ``label``, ``hole`` (bool), ``depth`` (components odd, holes even), ``parent`` (label), ``area`` (cv2.contourArea),
        ``count`` / ``segsum`` / ``score``: pixels, mask sum and score-map sum under the FILLED contour;
      lab: int32 [h+2, w+2] label image of the frame padded by one background pixel: 1..nf foreground (8-connected),
        nf+1.. background (4-connected), lab[0, 0] = the outside;
      parent: the nesting tree over labels (the outside is its own parent).

    Every sum but ``score`` is an integer and exact; ``score`` is summed in another order than ``contour_objects`` (and
    the device), so it agrees with them to rounding only."""
    from scipy import ndimage as ndi
    X = np.asarray(X, bool)
    h, w = X.shape
    P = np.pad(X, 1)
    fl, nf = ndi.label(P, np.ones((3, 3), int))
    bl, _ = ndi.label(~P, np.array([[0, 1, 0], [1, 1, 1], [0, 1, 0]]))
    lab = np.where(P, fl, bl + nf).astype(np.int32)
    flat = lab.ravel()
    outer = int(flat[0])
    n = int(flat.max()) + 1                                  # label 0 is unused
    # the parent of a set = the set of the pixel left of its first pixel in raster order
    labels, first = np.unique(flat, return_index=True)
    parent = np.zeros(n, np.int64)
    parent[labels] = flat[first - 1]
    parent[outer] = outer
    # depths by pointer jumping
    depth = (parent != np.arange(n)).astype(np.int64)
    anc = parent.copy()
    while np.any(depth[anc]):
        depth, anc = depth + depth[anc], anc[anc]
    # per-set sums over the frame
    inner = lab[1:-1, 1:-1].ravel()
    cnt = np.bincount(inner, minlength=n).astype(np.int64)
    seg = np.bincount(inner, weights=np.asarray(segmask, np.float64).ravel(), minlength=n).astype(np.int64)
    score = np.bincount(inner, weights=np.asarray(score_map, np.float64).ravel(), minlength=n)
    # the ring of a hole: the pixels of its parent component 4-adjacent to it, each counted once per hole
    fgpix = X.ravel()
    lf = inner[fgpix]
    pf = parent[lf]
    nbs = [lab[1:-1, :-2], lab[1:-1, 2:], lab[:-2, 1:-1], lab[2:, 1:-1]]
    nbs = [b.ravel()[fgpix] for b in nbs]
    sg_f = np.asarray(segmask, np.float64).ravel()[fgpix]
    sc_f = np.asarray(score_map, np.float64).ravel()[fgpix]
    rcnt, rseg, rscore = np.zeros(n, np.int64), np.zeros(n, np.int64), np.zeros(n)
    for j, b in enumerate(nbs):
        m = (b > nf) & (b != pf)
        for q in range(j):
            m &= b != nbs[q]
        rcnt += np.bincount(b[m], minlength=n)
        rseg += np.bincount(b[m], weights=sg_f[m], minlength=n).astype(np.int64)
        rscore += np.bincount(b[m], weights=sc_f[m], minlength=n)
    del nbs, lf, pf
    # L: pixel edges between a component and its parent (its outer border) or one of its holes (that hole's border)
    L = np.zeros(n, np.int64)
    for la, lb in ((lab[:, :-1], lab[:, 1:]), (lab[:-1, :], lab[1:, :])):
        fa, fb = la <= nf, lb <= nf
        e = fa != fb
        lfg = np.where(fa, la, lb)[e]
        lbg = np.where(fa, lb, la)[e]
        L += np.bincount(np.where(lbg == parent[lfg], lfg, lbg), minlength=n)
    # 2x2 windows with one foreground pixel and three pixels of one background set: n1 of the component when that set is
    # its parent, else n3 of that hole
    win = (lab[:-1, :-1], lab[:-1, 1:], lab[1:, :-1], lab[1:, 1:])
    nfg = sum((x <= nf).astype(np.int8) for x in win)
    one = nfg == 1
    ws = [x[one] for x in win]
    lfg = np.max([np.where(x <= nf, x, 0) for x in ws], axis=0)
    bmin = np.min([np.where(x <= nf, n, x) for x in ws], axis=0)
    bmax = np.max([np.where(x <= nf, 0, x) for x in ws], axis=0)
    same = bmin == bmax
    lfg, b = lfg[same], bmin[same]
    nw = np.bincount(np.where(b == parent[lfg], lfg, b), minlength=n)
    del win, nfg, one, ws
    # subtree totals, deepest level first: a filled contour covers its set and everything nested in it
    order = np.argsort(depth, kind="stable")[::-1]
    ds = depth[order]
    bounds = np.flatnonzero(np.diff(ds)) + 1
    for grp in np.split(order, bounds):
        if depth[grp[0]] == 0:
            continue
        p = parent[grp]
        np.add.at(cnt, p, cnt[grp])
        np.add.at(seg, p, seg[grp])
        np.add.at(score, p, score[grp])
    ids = np.delete(np.arange(1, n), outer - 1)
    hole = ids > nf
    B = (L[ids] - nw[ids]) / 2.0
    rec = {
        "label": ids, "hole": hole, "depth": depth[ids], "parent": parent[ids],
        "area": np.where(hole, cnt[ids] + B - 1, cnt[ids] - B - 1),
        "count": cnt[ids] + np.where(hole, rcnt[ids], 0),
        "segsum": seg[ids] + np.where(hole, rseg[ids], 0),
        "score": score[ids] + np.where(hole, rscore[ids], 0.0),
    }
    return rec, lab, parent, nf


def remove_invalid_objects_fast(cfg, alpha, segmask=None, return_records=False):
    """``remove_invalid_objects`` on ``contour_records``: the same result (tests/test_oracle_objects_fast.py), fast
    enough for 1080p and 4K frames.  With ``return_records`` also the records, plus per contour ``saliency``,
    ``consensus``, ``valid`` and the decision margins: ``sal_margin`` = relative distance of the saliency from
    saliency_thr and from 10 * saliency_thr (the nearer one), ``con_margin`` = relative distance of the consensus from
    consensus_thr.  Only the saliency is a floating-point sum whose order matters (the consensus is an integer sum
    divided the same way everywhere), so ``sal_margin`` of the contours with area >= 100 bounds what summation order
    could flip."""
    saliency_thr = cfg['objectremoval']['saliency_thr']
    consensus_thr = cfg['objectremoval']['consensus_thr']
    if segmask is None:
        segmask = alpha
    h, w = alpha.shape
    rec, lab, parent, nf = contour_records(alpha > 0, segmask, build_score_map(h, w, cfg))
    saliency = rec["score"] / float(h * w)
    consensus = rec["segsum"] / rec["count"] / 255.
    valid = ~(rec["area"] < 100) & (((saliency > saliency_thr) & (consensus > consensus_thr)) | (saliency > saliency_thr * 10))
    # painted: the pixel's set or one of its ancestors is a valid contour (pointer jumping up the tree) ...
    n = parent.size
    flag = np.zeros(n, bool)
    flag[rec["label"]] = valid
    anc = parent.copy()
    while True:
        flag = flag | flag[anc]
        nxt = anc[anc]
        if np.array_equal(nxt, anc):
            break
        anc = nxt
    vhole = np.zeros(n, bool)
    vhole[rec["label"][rec["hole"] & valid]] = True
    keep = flag[lab[1:-1, 1:-1]]
    # ... or it is on the ring of a valid hole
    for b in (lab[1:-1, :-2], lab[1:-1, 2:], lab[:-2, 1:-1], lab[2:, 1:-1]):
        keep |= vhole[b]
    out = np.where(keep & (alpha > 0), alpha, 0).astype(alpha.dtype)
    if not return_records:
        return out
    rec.update(saliency=saliency, consensus=consensus, valid=valid,
               sal_margin=np.minimum(np.abs(saliency - saliency_thr) / saliency_thr,
                                     np.abs(saliency - 10 * saliency_thr) / (10 * saliency_thr)),
               con_margin=np.abs(consensus - consensus_thr) / consensus_thr)
    return out, rec


def decision_margin(rec):
    """the smallest ``sal_margin`` over the contours whose scores decide anything (area >= 100); inf without any"""
    m = rec["sal_margin"][~(rec["area"] < 100)]
    return float(m.min()) if m.size else float("inf")


def remove_invalid_objects(cfg, alpha, segmask=None, objs=None):
    """unscreen/utils/maskprocess.py:77-152 on the closed-form contour model above (does not mutate ``alpha``).
    ``objs``: contour_objects(alpha > 0) when the caller already has it."""
    saliency_thr = cfg['objectremoval']['saliency_thr']
    consensus_thr = cfg['objectremoval']['consensus_thr']
    if segmask is None:
        segmask = alpha
    h, w = alpha.shape
    score_map = build_score_map(h, w, cfg)
    valid = np.zeros((h, w), bool)
    for fill, area in (contour_objects(alpha > 0) if objs is None else objs):
        if area < 100:
            continue
        saliency = score_map[fill].sum() / float(h * w)
        consensus = segmask[fill].astype(np.float64).mean() / 255.
        if (saliency > saliency_thr and consensus > consensus_thr) or saliency > saliency_thr * 10:
            valid |= fill
    out = alpha.copy()
    out[~valid] = 0
    return out
