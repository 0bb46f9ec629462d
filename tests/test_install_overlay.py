"""video_unscreen_b200.install(): with the reference checkout importable it must OVERLAY the reference package (hot-path
names replaced, everything else the reference's), so that the exact import blocks of the reference's pipeline scripts
resolve; without it, it aliases the mirror.  Runs in a subprocess (install() edits sys.modules); no GPU needed: nothing
is called, only imported."""
import os
import subprocess
import sys
import textwrap

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.environ.get("UNSCREEN_REFERENCE", "")   # a checkout of AnyiRao/video_unscreen; the overlay tests skip without it
HAVE_REF = bool(REF) and os.path.isdir(os.path.join(REF, "unscreen"))

SHIM = """
import sys, types
import numpy as np
np.float = float; np.int = int            # the reference predates numpy 1.24 (SURVEY.md section 8c shim)
for n in ("mmcv", "matplotlib", "matplotlib.pyplot"):   # absent in this container, unused on the arithmetic path
    sys.modules.setdefault(n, types.ModuleType(n))
sys.modules["matplotlib"].pyplot = sys.modules["matplotlib.pyplot"]
sys.path.insert(0, %r)
"""


def _run(code):
    r = subprocess.run([sys.executable, "-c", textwrap.dedent(code)], capture_output=True, text=True, cwd=ROOT, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    return r.stdout


@pytest.mark.skipif(not HAVE_REF, reason="reference checkout not present (set UNSCREEN_REFERENCE)")
def test_overlay_keeps_the_reference_scripts_importable():
    out = _run((SHIM % ROOT) + f"""
sys.path.insert(0, {REF!r})
import video_unscreen_b200 as vu
vu.install()
import video_unscreen_b200.unscreen.utils as mine
import video_unscreen_b200.unscreen.colorfiltering as mine_cf
import video_unscreen_b200.unscreen.trimap as mine_tri

# tools/unscreen/green.py:11-18 (unscreen.binseg needs torchvision.models.utils, gone from this container's torchvision:
# it fails the same way without install(), so it is imported guardedly)
from unscreen.colorfiltering import ColorFilteringAgent
from unscreen.trimap import TrimapAgent
from unscreen.utils import (exist_foreground, color_correct,
                            get_fg, parallel_read_img,
                            remove_invalid_objects,
                            save_img, save_video)
from unscreen.vmatting import VMattingAgent
# tools/unscreen/bg.py:13-19
from unscreen.stm import STMAgent
from unscreen.utils import (dilate_mask, exist_foreground, get_bg, get_fg,
                            parallel_read_img, regionfill,
                            remove_invalid_objects, save_img, save_video)
# tools/unscreen/bg_offline.py:13-20
from unscreen.utils import (adaptive_resize, build_score_map, dilate_mask,
                            get_bg, get_fg,
                            exist_foreground, parallel_read_img, regionfill,
                            remove_invalid_objects, save_img, save_video)
# tools/replace/replace.py:14-15
from unscreen.utils import (adaptive_resize, get_center, rescale_fg,
                            return_date, shift_fg)
from unscreen.bgmodel import BackgroundAgent

import unscreen, unscreen.utils.maskprocess as ref_mp
assert unscreen.__file__.startswith({REF!r}), unscreen.__file__
# hot-path names are the B200 mirror's ...
for name in ("get_fg", "get_bg", "dilate_mask", "exist_foreground", "color_correct", "adaptive_resize", "rescale_fg",
             "shift_fg", "remove_invalid_objects", "build_score_map"):
    assert globals()[name] is getattr(mine, name), name
assert ColorFilteringAgent is mine_cf.ColorFilteringAgent and TrimapAgent is mine_tri.TrimapAgent
# ... also inside the reference's own modules (remove_invalid_objects calls its module's dilate_mask)
assert ref_mp.dilate_mask is mine.dilate_mask
assert unscreen.utils.temporal_median is mine.temporal_median
# ... and everything else is still the reference's
for f in (parallel_read_img, save_img, save_video, get_center, return_date):
    assert f.__module__.startswith("unscreen."), (f, f.__module__)
assert regionfill is mine.regionfill
assert VMattingAgent.__module__ == "unscreen.vmatting.agent" and STMAgent.__module__.startswith("unscreen.stm")
import unscreen.bgmodel.agent as ref_bg, video_unscreen_b200.unscreen.bgmodel as mine_bg
assert BackgroundAgent is mine_bg.BackgroundAgent and ref_bg.BackgroundAgent is BackgroundAgent
assert BackgroundAgent(input_long_side=100).pcov_ksize == 5
assert "unscreen.utils.fgfuncs.get_fg" in vu.installed_names()
print("overlay ok", len(vu.installed_names()))
""")
    assert "overlay ok" in out


@pytest.mark.skipif(not HAVE_REF, reason="reference checkout not present (set UNSCREEN_REFERENCE)")
def test_overlay_io_is_opt_in():
    out = _run((SHIM % ROOT) + f"""
sys.path.insert(0, {REF!r})
import video_unscreen_b200 as vu
vu.install(io=True)
from unscreen.utils import parallel_read_img, save_img, save_video
import unscreen.utils.fileio as ref_io
assert parallel_read_img.__module__ == "video_unscreen_b200.unscreen.utils.fileio" and ref_io.save_img is save_img
assert save_video.__module__.startswith("unscreen.")          # mmcv / ffmpeg: the reference's
print("io ok")
""")
    assert "io ok" in out


def test_alias_mode_without_the_reference():
    out = _run(f"""
import sys
sys.path.insert(0, {ROOT!r})
sys.path = [p for p in sys.path if not p.rstrip('/').endswith('reference')]
import video_unscreen_b200 as vu
vu.install()
from unscreen.colorfiltering import ColorFilteringAgent
from unscreen.trimap import TrimapAgent
from unscreen.bgmodel import BackgroundAgent
from unscreen.utils import (dilate_mask, erode_mask, exist_foreground, get_outer_boundary, is_pixel_inrange, get_fg,
                            get_bg, get_fg_naive, composite_fgbg, fuse_fgbg, get_target_size, adaptive_resize,
                            color_correct, shift_fg, rescale_fg, temporal_median, masked_temporal_mean)
assert ColorFilteringAgent.__module__.startswith("video_unscreen_b200.")
assert vu.installed_names() == ["*"]
print("alias ok")
""")
    assert "alias ok" in out
