"""mask processing (reference: unscreen/utils/maskprocess.py)."""
import torch

from ... import _lib, ops
from ..._io import back, to_dev

import numpy as np

__all__ = ["dilate_mask", "erode_mask", "exist_foreground", "get_outer_boundary", "remove_invalid_objects", "get_score_map",
           "build_score_map"]


def _morph(mask, kernelsize, iters, op):
    t, as_np = to_dev(mask)
    if t.ndim == 3 and t.shape[-1] == 3:
        # the reference also feeds 3-channel masks (bg_offline.py:116): per-channel morphology
        planes = t.permute(2, 0, 1).contiguous()
        out = ops.morph(planes, kernelsize, iters, op).permute(1, 2, 0).contiguous()
    else:
        out = ops.morph(t, kernelsize, iters, op)
    return back(out, as_np)


def dilate_mask(mask, kernelsize=5, iters=10):
    """reference maskprocess.py:7-19."""
    return _morph(mask, kernelsize, iters, _lib.DILATE)


def erode_mask(mask, kernelsize=5, iters=10):
    """reference maskprocess.py:22-34."""
    return _morph(mask, kernelsize, iters, _lib.ERODE)


def exist_foreground(mask, fg_exist_thr):
    """reference maskprocess.py:56-60: count(mask >= 128) > thr*h*w (strict)."""
    t, _ = to_dev(mask)
    h, w = t.shape
    n = int(ops.count_cmp(t, _lib.CMP_GE, 128).item())
    return bool(n > fg_exist_thr * h * w)


def get_outer_boundary(mask, kernelsize=7, iters=10):
    """reference maskprocess.py:63-74 (uint8 subtraction wraps; the clip is a no-op)."""
    t, as_np = to_dev(mask)
    d = ops.dilate(t, kernelsize, iters)
    return back(ops.sub_wrap(d, t), as_np)


def get_score_map(map_size, center):
    """reference maskprocess.py:155-178: 1 at ``center`` (a ratio of the size), falling linearly to 0 at the borders"""
    score_map = np.ones(map_size, np.float64)
    h, w = map_size
    y, x = int(h * center[0]), int(w * center[1])
    score_map[:, x:w] = np.linspace(0, 1, w - x)[np.newaxis, ...]**2
    score_map[:, 0:x] = np.linspace(1, 0, x)[np.newaxis, ...]**2
    score_map[y:h] += np.linspace(0, 1, h - y)[..., np.newaxis]**2
    score_map[0:y] += np.linspace(1, 0, y)[..., np.newaxis]**2
    score_map = np.sqrt(score_map)
    score_map = (score_map.max() - score_map) / score_map.max()
    return score_map


def build_score_map(h, w, config):
    """reference maskprocess.py:181-189."""
    centers = config['objectremoval']['score_map_center']
    return get_score_map((h, w), centers['landscape'] if w > h else centers['portrait'])


_SCORE_MAPS = {}


def _score_map_dev(h, w, cfg, device):
    centers = cfg['objectremoval']['score_map_center']
    center = tuple(centers['landscape'] if w > h else centers['portrait'])
    key = (h, w, center, str(device))
    if key not in _SCORE_MAPS:
        _SCORE_MAPS[key] = torch.from_numpy(get_score_map((h, w), center)).to(device)
    return _SCORE_MAPS[key]


def remove_invalid_objects(cfg, alpha, segmask=None, saliency_thr=0.001, consensus_thr=0.5, score_map=None,
                           score_map_center=(3. / 5, 1. / 2), max_objects=16384):
    """reference maskprocess.py:77-152: clear every object (contour of cv2.findContours) whose saliency or consensus score
    fails.  As in the reference the thresholds and the score map come from ``cfg['objectremoval']`` (the keyword arguments
    of the same name are ignored there too).  ``alpha`` may be [H,W] or a clip [N,H,W]; it is not modified.  Frames with
    more than ``max_objects`` contours are redone with a larger table."""
    saliency_thr = cfg['objectremoval']['saliency_thr']
    consensus_thr = cfg['objectremoval']['consensus_thr']
    a, as_np = to_dev(alpha)
    s = a if segmask is None else to_dev(segmask)[0]
    h, w = a.shape[-2:]
    sm = _score_map_dev(h, w, cfg, a.device)
    while True:
        out, status = ops.remove_invalid_objects(a, s, sm, saliency_thr, consensus_thr, max_objects)
        worst = int(status.max().item())
        if worst <= max_objects:
            break
        max_objects = worst
    return back(out, as_np)
