"""ctypes binding of the C ABI in include/gf_attn.h (libgf_attn.so).

This is the binding a maintainer of the reference would add inside ``transformer_layer`` (see INTEGRATION.md):
raw device pointers and sizes only, no torch types cross the boundary.  There is no fallback: if the library
cannot be loaded, or a call fails, a RuntimeError is raised.
"""
from __future__ import annotations

import ctypes
from ctypes import c_int, c_int32, c_size_t, c_void_p, c_char_p, POINTER, byref
from typing import Optional

from ._build import LIB_PATH, build_extension

GF_OK = 0
NORM = {None: 0, "none": 0, "layer": 1, "instance": 2, "batch": 3}
INTEGRATION = {"mul": 0, "add": 1, "both": 2}
FLAG_FP32_EXACT = 1
FLAG_CENTROIDS_IN = 2
FLAG_TABLES_READY = 4
FLAG_IMG2LTNT = 8
FLAG_CENTROIDS_INIT = 16
PATH_NAMES = {0: "none", 1: "simt_fp32", 2: "tcgen05_tf32"}

WEIGHT_FIELDS = ("wq", "bq", "wpq", "wk", "bk", "wpk", "wv", "bv", "wo", "bo", "pos_latent",
                 "wq2", "bq2", "wpq2", "wk2", "bk2", "wpk2", "wv2", "bv2", "wkc", "wcq", "wi2l", "bi2l")

# every symbol include/gf_attn.h declares (tests check the .so exports each of them)
EXPORTS = ("gf_attn_abi_version", "gf_last_error", "gf_attn_last_path", "gf_attn_folded_floats",
           "gf_attn_fold_weights", "gf_attn_workspace_bytes", "gf_attn_prologue", "gf_attn_simplex_fwd",
           "gf_attn_duplex_fwd", "gf_attn_norm_stats", "gf_attn_launch_count",
           "gf_attn_simplex_fwd_ex", "gf_attn_duplex_fwd_ex", "gf_attn_prologue_ex", "gf_attn_simplex_bwd", "gf_attn_last_centroid_path", "gf_attn_debug_layout",
           "gf_attn_prologue_batch", "gf_attn_tc_eligible", "gf_attn_simplex_bwd_ex", "gf_attn_dropout_mask",
           "gf_attn_centroid_recompute", "gf_attn_centroid_bwd")
# include/gf_ops.h
OPS_EXPORTS = ("gf_chan_scale_nhwc", "gf_blur_up_nhwc", "gf_upsample2x_nchw", "gf_bias_act_nhwc", "gf_demod_coef", "gf_torgb_nhwc", "gf_fir4_nhwc", "gf_blur_up_phases_nhwc", "gf_torgb_scale_nhwc", "gf_mapping_fwd", "gf_conv3x3_pack_weights", "gf_conv3x3_nhwc_tf32", "gf_demod_coef_batch", "gf_conv3x3_nhwc_tf32_ex", "gf_conv3x3_last_variant")


class GfAttnDesc(ctypes.Structure):
    _fields_ = [(n, c_int32) for n in ("B", "H", "W", "C", "k", "D", "heads", "norm", "integration",
                                       "pos_dim", "duplex", "flags")]


class GfAttnWeights(ctypes.Structure):
    _fields_ = [(n, c_void_p) for n in WEIGHT_FIELDS]


class GfAttnPostop(ctypes.Structure):
    _fields_ = [("bias", c_void_p), ("noise", c_void_p), ("strength", c_void_p), ("noise_bstride", ctypes.c_longlong),
                ("act", c_int32), ("gain", ctypes.c_float), ("in_scale", c_void_p), ("post_scale", c_void_p),
                ("in_scale_ld", c_int32), ("post_scale_ld", c_int32),
                ("rgb_w", c_void_p), ("rgb_bias", c_void_p), ("rgb_out", c_void_p),
                ("att_dp", ctypes.c_float), ("dp_salt", ctypes.c_uint32), ("dp_state", c_void_p)]


_lib: Optional[ctypes.CDLL] = None


def load() -> ctypes.CDLL:
    """Load (building first if missing/stale) libgf_attn.so.  Raises on failure -- never falls back."""
    global _lib
    if _lib is not None:
        return _lib
    import os
    alt = os.environ.get("GF_ATTN_LIB")          # A/B benchmarking of two builds of the same sources (tools/ab_build.sh)
    if alt:
        lib = ctypes.CDLL(alt)
    else:
        try:
            build_extension()
        except Exception as e:  # nvcc missing is fine as long as a prebuilt .so is present
            if not LIB_PATH.exists():
                raise RuntimeError(f"libgf_attn.so is missing and could not be built: {e}") from e
        lib = ctypes.CDLL(str(LIB_PATH))
    lib.gf_attn_abi_version.restype = c_int
    lib.gf_last_error.restype = c_char_p
    lib.gf_attn_last_path.restype = c_int
    lib.gf_attn_folded_floats.argtypes = [POINTER(GfAttnDesc), POINTER(c_size_t)]
    lib.gf_attn_workspace_bytes.argtypes = [POINTER(GfAttnDesc), POINTER(c_size_t)]
    lib.gf_attn_fold_weights.argtypes = [POINTER(GfAttnDesc), POINTER(GfAttnWeights), c_void_p, c_void_p]
    lib.gf_attn_prologue.argtypes = [POINTER(GfAttnDesc), c_void_p, c_void_p, c_void_p, c_void_p]
    lib.gf_attn_simplex_fwd.argtypes = [POINTER(GfAttnDesc), c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]
    lib.gf_attn_duplex_fwd.argtypes = [POINTER(GfAttnDesc), c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                       c_void_p, c_void_p, c_void_p]
    lib.gf_attn_norm_stats.argtypes = [POINTER(GfAttnDesc), c_void_p, c_void_p, c_void_p]
    lib.gf_attn_debug_layout.argtypes = [POINTER(GfAttnDesc), POINTER(ctypes.c_longlong), c_int]
    lib.gf_attn_prologue_ex.argtypes = [POINTER(GfAttnDesc), c_void_p, c_void_p, c_void_p, POINTER(GfAttnPostop), c_void_p]
    lib.gf_attn_simplex_fwd_ex.argtypes = [POINTER(GfAttnDesc), c_void_p, c_void_p, c_void_p, c_void_p, POINTER(GfAttnPostop), c_void_p]
    lib.gf_attn_duplex_fwd_ex.argtypes = [POINTER(GfAttnDesc), c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                          c_void_p, c_void_p, POINTER(GfAttnPostop), c_void_p]
    lib.gf_attn_prologue_batch.argtypes = [c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]
    lib.gf_attn_simplex_bwd.argtypes = [POINTER(GfAttnDesc)] + [c_void_p] * 11
    lib.gf_attn_simplex_bwd_ex.argtypes = [POINTER(GfAttnDesc)] + [c_void_p] * 10 + [ctypes.c_float, ctypes.c_uint32, c_void_p, c_void_p, c_void_p]
    lib.gf_attn_centroid_recompute.argtypes = [POINTER(GfAttnDesc)] + [c_void_p] * 8
    lib.gf_attn_centroid_bwd.argtypes = [POINTER(GfAttnDesc)] + [c_void_p] * 10
    lib.gf_attn_dropout_mask.argtypes = [POINTER(GfAttnDesc), ctypes.c_float, ctypes.c_uint32, c_void_p, c_void_p, c_void_p]
    lib.gf_chan_scale_nhwc.argtypes = [c_void_p, c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_void_p]
    lib.gf_blur_up_nhwc.argtypes = [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, ctypes.c_float, c_void_p]
    lib.gf_upsample2x_nchw.argtypes = [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p]
    lib.gf_bias_act_nhwc.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, ctypes.c_longlong, c_int, c_int, c_int,
                                     c_int, ctypes.c_float, c_void_p]
    lib.gf_demod_coef.argtypes = [c_void_p, c_int, c_void_p, c_void_p, c_int, c_int, c_int, ctypes.c_float, c_void_p]
    lib.gf_blur_up_phases_nhwc.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int,
                                           ctypes.c_float, c_void_p]
    lib.gf_fir4_nhwc.argtypes = [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, ctypes.c_float, c_void_p]
    lib.gf_torgb_scale_nhwc.argtypes = [c_void_p, c_void_p, c_void_p, c_int, c_void_p, ctypes.c_float, c_void_p, c_void_p, c_int, c_void_p,
                                        c_int, c_int, c_int, c_void_p]
    lib.gf_mapping_fwd.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, ctypes.c_float, c_void_p, c_int, c_int, c_int, c_int, c_void_p]
    lib.gf_conv3x3_pack_weights.argtypes = [c_void_p, c_void_p, c_int, c_int, ctypes.c_float, c_void_p]
    lib.gf_conv3x3_nhwc_tf32.argtypes = [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p]
    lib.gf_conv3x3_nhwc_tf32_ex.argtypes = [c_void_p, c_void_p, c_void_p] + [c_int] * 8 + [c_void_p]
    lib.gf_conv3x3_last_variant.argtypes = [POINTER(c_int)] * 3
    lib.gf_demod_coef_batch.argtypes = [c_void_p, c_int, c_int, ctypes.c_float, c_void_p]
    lib.gf_torgb_nhwc.argtypes = [c_void_p, c_void_p, c_void_p, c_int, c_void_p, ctypes.c_float, c_void_p, c_int, c_int, c_int, c_void_p]
    for name in OPS_EXPORTS:
        getattr(lib, name).restype = c_int
    for name in EXPORTS:
        fn = getattr(lib, name)
        if name not in ("gf_last_error", "gf_attn_launch_count"):
            fn.restype = c_int
    lib.gf_attn_launch_count.restype = ctypes.c_longlong
    lib.gf_attn_tc_eligible.argtypes = [POINTER(GfAttnDesc)]
    if lib.gf_attn_abi_version() != 2:
        raise RuntimeError("libgf_attn.so ABI version mismatch")
    _lib = lib
    return lib


class GfDemodJob(ctypes.Structure):
    """gf_demod_job of include/gf_ops.h."""
    _fields_ = [("styles", c_void_p), ("wsq", c_void_p), ("d", c_void_p), ("s_ld", ctypes.c_int32), ("O", ctypes.c_int32),
                ("I", ctypes.c_int32), ("pad_", ctypes.c_int32)]


DEMOD_MAX_JOBS = 32


def check(rc: int, what: str) -> None:
    if rc != GF_OK:
        msg = load().gf_last_error().decode("utf-8", "replace")
        raise RuntimeError(f"{what} failed (gf_status {rc}): {msg}")


def make_desc(B, H, W, C, k, D, *, heads=1, norm="layer", integration="mul", pos_dim=0, duplex=False, flags=0) -> GfAttnDesc:
    if norm not in NORM:
        raise ValueError(f"unknown norm {norm!r}")
    if integration not in INTEGRATION:
        raise ValueError(f"unknown integration {integration!r}")
    return GfAttnDesc(B, H, W, C, k, D, heads, NORM[norm], INTEGRATION[integration], pos_dim, int(duplex), flags)    # duplex: 0 or the number of k-means iterations


def folded_floats(desc: GfAttnDesc) -> int:
    out = c_size_t(0)
    check(load().gf_attn_folded_floats(byref(desc), byref(out)), "gf_attn_folded_floats")
    return out.value


def workspace_bytes(desc: GfAttnDesc) -> int:
    out = c_size_t(0)
    check(load().gf_attn_workspace_bytes(byref(desc), byref(out)), "gf_attn_workspace_bytes")
    return out.value


def launch_count() -> int:
    return int(load().gf_attn_launch_count())


def last_centroid_path() -> str:
    return PATH_NAMES.get(load().gf_attn_last_centroid_path(), "?")


def last_path() -> str:
    return PATH_NAMES.get(load().gf_attn_last_path(), "?")


def conv3x3_last_variant() -> tuple:
    """(version, bn, mt) of the convolution kernel the last gf_conv3x3_nhwc_tf32[_ex] call on this thread launched."""
    v = (c_int(0), c_int(0), c_int(0))
    check(load().gf_conv3x3_last_variant(*(byref(i) for i in v)), "gf_conv3x3_last_variant")
    return tuple(i.value for i in v)
