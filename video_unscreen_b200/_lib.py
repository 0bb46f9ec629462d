"""ctypes binding of libvu_b200.so (the C ABI declared in include/vu_b200.h).

The library is the product: if it is missing or a call fails, this module
raises -- there is no CPU or PyTorch fallback behind it.
"""
import ctypes
import os
import re

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libvu_b200.so")
HEADER_PATH = os.path.join(os.path.dirname(_HERE), "include", "vu_b200.h")

VU_OK = 0
DILATE, ERODE = 0, 1
CMP_GE, CMP_GT, CMP_LT, CMP_EQ, CMP_NE = range(5)
PATCH_NONE, PATCH_ALPHA_LT128, PATCH_ALPHA_EQ0 = range(3)
BLEND_NAIVE, BLEND_FUSE, BLEND_COMPOSITE, BLEND_REPLACE = range(4)
ERR_UNSUPPORTED = -2   # enum vu_status: VU_ERR_UNSUPPORTED

_p = ctypes.c_void_p
_i = ctypes.c_int
_i64 = ctypes.c_int64
_sz = ctypes.c_size_t
_f = ctypes.c_float
_d = ctypes.c_double
_i3 = ctypes.POINTER(ctypes.c_int32)

# name -> (restype, argtypes); must list every function of include/vu_b200.h
SIGNATURES = {
    "vu_abi_version": (_i, []),
    "vu_status_string": (ctypes.c_char_p, [_i]),
    "vu_last_cuda_error": (ctypes.c_char_p, []),
    "vu_launch_count": (ctypes.c_uint64, []),
    "vu_bgr2hsv_u8": (_i, [_p, _p, _i64, _p]),
    "vu_hsv2bgr_u8": (_i, [_p, _p, _i64, _p]),
    "vu_bgr2gray_u8": (_i, [_p, _p, _i64, _p]),
    "vu_inrange_color": (_i, [_p, _i64, _i3, _i3, _p, _p]),
    "vu_inrange_image": (_i, [_p, _p, _i64, _i64, _i3, _p, _p]),
    "vu_morph_workspace_bytes": (_sz, [_i, _i, _i, _i, _i]),
    "vu_morph_u8": (_i, [_p, _p, _i, _i, _i, _i, _i, _i, _p, _sz, _p]),
    "vu_cross_chain_u8": (_i, [_p, _p, _i, _i, _i, _i, _i3, _i3, _p, _d, _p]),
    "vu_trimap_core_u8": (_i, [_p, _p, _i, _i, _i, _i, _p]),
    "vu_resize_linear_u8": (_i, [_p, _i, _i, _i, _i, _p, _i, _i, _p]),
    "vu_resize_nearest_u8": (_i, [_p, _i, _i, _i, _i, _p, _i, _i, _p]),
    "vu_shift_u8": (_i, [_p, _p, _i, _i, _i, _i, _f, _f, _p]),
    "vu_rescale_cubic_u8": (_i, [_p, _p, _i, _i, _i, _i, _d, _p]),
    "vu_color_correct_workspace_bytes": (_sz, [_i, _i, _i]),
    "vu_color_correct": (_i, [_p, _p, _p, _i, _i, _i, _i, _i, _p, _d, _p, _p, _sz, _p]),
    "vu_color_correct_frames": (_i, [_p, _p, _i, _i, _i, _i, _i, _p, _d, _p, _p, _sz, _p]),
    "vu_count_cmp_u8": (_i, [_p, _i, _i64, _i, _i, _p, _p]),
    "vu_count_and_u8": (_i, [_p, _p, _i, _i64, _p, _p]),
    "vu_mask_clear_where": (_i, [_p, _p, _p, _i64, _p]),
    "vu_mask_set128_where": (_i, [_p, _p, _p, _i64, _p]),
    "vu_mask_and01": (_i, [_p, _p, _p, _i64, _p]),
    "vu_trimap_bits_workspace_bytes": (ctypes.c_size_t, [_i, _i, _i]),
    "vu_trimap_bits": (_i, [_p, _p, _p, _i, _i, _i, _i, _i, _i, _p, _p, ctypes.c_size_t, _p]),
    "vu_trimap_bits_packed": (_i, [_p, _p, _p, _i, _i, _i, _i, _i, _i, _p, _p, ctypes.c_size_t, _p]),
    "vu_cf_alpha_up_fuzzy": (_i, [_p, _i, _i, _i, _i, _i, _p, _p, _p, _i3, _i3, _p, _p, _p, _p, _p, _p, _p, _p]),
    "vu_trimap_classify": (_i, [_p, _p, _p, _i64, _p]),
    "vu_trimap_snap": (_i, [_p, _i64, _p, _p]),
    "vu_ratio_flags": (_i, [_p, _i, _d, _p, _p]),
    "vu_cf_degenerate_flags": (_i, [_p, _p, _i, _i, ctypes.c_uint64, ctypes.c_uint64, _p, _p]),
    "vu_count_gt_lt_u8": (_i, [_p, _i, _i64, _i, _p, _p]),
    "vu_select_frames": (_i, [_p, _p, _p, _i, _i64, _p, _p]),
    "vu_set128_unflagged": (_i, [_p, _p, _p, _i, _i64, _p, _p]),
    "vu_cf_samples_workspace_bytes": (ctypes.c_size_t, [_i]),
    "vu_cf_samples": (_i, [_p, _p, _i, _i, _i, _i, _i, _i, _i, _p, _i, _p, _p, _p, ctypes.c_size_t, _p]),
    "vu_cf_lowres": (_i, [_p, _p, _i, _i, _i, _i, _i, _p, _p, _p, _p, _p]),
    "vu_resize_up_u8": (_i, [_p, _i, _i, _i, _p, _i, _i, _i, _p, _p, _p, _p, _p]),
    "vu_fuzzy_count": (_i, [_p, _p, _i, _i64, _i3, _i3, _p, _p, _p]),
    "vu_trimap_src_lo": (_i, [_p, _p, _p, _i, _i, _i, _i, _i, _p, _p]),
    "vu_cf_alpha_u8": (_i, [_p, _i64, _p, _p, _p]),
    "vu_cf_build_lut3d": (_i, [_p, _p, _p]),
    "vu_cf_alpha_lut3d_u8": (_i, [_p, _i64, _p, _p, _p]),
    "vu_cf_threshold_stats": (_i, [_p, _p, _i, _i64, _p, _p]),
    "vu_cf_threshold_apply": (_i, [_p, _i, _i64, _p, _d, _p, _p]),
    "vu_mask_bbox": (_i, [_p, _i, _i, _p, _p]),
    "vu_masked_sum3": (_i, [_p, _p, _i64, _p, _p]),
    "vu_pcov_round": (_i, [_p, _p, _i, _i, _i, _i, _i, _p, _p, _p, _i, _p]),
    "vu_remove_objects_workspace_bytes": (ctypes.c_size_t, [_i, _i, _i, _i]),
    "vu_remove_invalid_objects": (_i, [_p, _p, _p, _i, _i, _i, _d, _d, _p, _p, _p, ctypes.c_size_t, _i, _p]),
    "vu_regionfill_workspace_bytes": (_sz, [_i, _i, _i]),
    "vu_regionfill_f64": (_i, [_p, _p, _i, _i, _i, _d, _i, _d, _p, _sz, _p, _p, _p]),
    "vu_resize_linear_f64": (_i, [_p, _i, _i, _i, _p, _i, _i, _d, _d, _p, _p, _p]),
    "vu_planar_rgb_to_bgr": (_i, [_p, _p, _i64, _p]),
    "vu_bgr_to_planar_rgb": (_i, [_p, _p, _i64, _p]),
    "vu_get_fg": (_i, [_p, _p, _p, _i64, _i64, _i, _p, _p, _p]),
    "vu_get_bg": (_i, [_p, _p, _i64, _p, _p]),
    "vu_blend": (_i, [_i, _p, _p, _i, _p, _i64, _i64, _p, _p]),
    "vu_fuse_bg": (_i, [_p, _p, _i64, _i64, _f, _f, _p, _p]),
    "vu_bgdiff_gray": (_i, [_p, _p, _i64, _i64, _i, _p, _p]),
    "vu_gate": (_i, [_p, _p, _i64, _p, _p]),
    "vu_bgdiff_gate": (_i, [_p, _p, _p, _i, _i, _i, _i, _i, _p, _p]),
    "vu_bgstep_frames": (_i, [_p, _p, _p, _i, _i, _i, _i, _i, _p, _p, _p, _i, _p]),
    "vu_binarise": (_i, [_p, _i64, _i, _p, _p]),
    "vu_sub_wrap_u8": (_i, [_p, _p, _i64, _p, _p]),
    "vu_temporal_median_u8": (_i, [_p, _i, _i64, _p, _p]),
    "vu_temporal_median_workspace_bytes": (ctypes.c_size_t, [_i, _i64]),
    "vu_temporal_median_u8_ws": (_i, [_p, _i, _i64, _p, _p, ctypes.c_size_t, _p]),
    "vu_masked_temporal_mean": (_i, [_p, _p, _i, _i64, _i, _p, _p, _p]),
    "vu_masked_temporal_mean_dilate32": (_i, [_p, _p, _i, _i, _i, _i, _p, _p, _p]),
    "vu_median_accum_bytes": (_sz, [_i64]),
    "vu_median_accum_reset": (_i, [_p, _i64, _p]),
    "vu_median_accum_add_u8": (_i, [_p, _i64, _p, _i, _i, _p]),
    "vu_median_accum_finish_u8": (_i, [_p, _i64, _i, _p, _p]),
    "vu_masked_mean_accum_bytes": (_sz, [_i, _i]),
    "vu_masked_mean_accum_reset": (_i, [_p, _i, _i, _p]),
    "vu_masked_mean_accum_add_dilate32": (_i, [_p, _p, _p, _i, _i, _i, _p]),
    "vu_masked_mean_accum_add": (_i, [_p, _p, _p, _i, _i64, _p]),
    "vu_masked_mean_accum_finish": (_i, [_p, _i64, _i, _p, _p, _p]),
}


def declared_symbols(header_path=HEADER_PATH):
    """every function name declared in the public header"""
    text = open(header_path).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(vu_[a-z0-9_]+)\s*\(", text)))


class VuError(RuntimeError):
    pass


_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: build it with `python __graft_entry__.py` "
                "(nvcc, sm_100a). There is no fallback path.")
        handle = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)  # AttributeError if the .so lacks a declared symbol
            fn.restype = res
            fn.argtypes = args
        if handle.vu_abi_version() != 1:
            raise ImportError("libvu_b200.so ABI version mismatch")
        _lib = handle
    return _lib


def check(status):
    if status != VU_OK:
        L = lib()
        msg = L.vu_status_string(status).decode()
        if status == -4:
            msg += ": " + L.vu_last_cuda_error().decode()
        raise VuError(f"libvu_b200 call failed ({status}): {msg}")


def i3(values):
    return (ctypes.c_int32 * 3)(*[int(v) for v in values])
