"""ctypes binding of librsb200.so (the C ABI declared in include/rsb200.h).

The library is built in-tree by `__graft_entry__.build()` / `robosat_b200/csrc/build.sh`.
There is no CPU fallback: if the shared object is missing, or no sm_100 device is usable,
every compute entry point raises `RsbError`.
"""

import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "librsb200.so")

RSB_MAX_SEGS = 16
RSB_MAX_SRCS = 4


class RsbError(RuntimeError):
    pass


class ConvSrc(ctypes.Structure):
    _fields_ = [
        ("ptr", ctypes.c_void_p),
        ("pitch_w", ctypes.c_int64),
        ("pitch_h", ctypes.c_int64),
        ("pitch_n", ctypes.c_int64),
        ("C", ctypes.c_int32),
        ("W", ctypes.c_int32),
        ("H", ctypes.c_int32),
        ("N", ctypes.c_int32),
        ("plane", ctypes.c_int64),
    ]


class ConvSeg(ctypes.Structure):
    _fields_ = [("src", ctypes.c_int32), ("dh", ctypes.c_int32), ("dw", ctypes.c_int32), ("cblocks", ctypes.c_int32)]


class ConvDesc(ctypes.Structure):
    _fields_ = [
        ("nsrc", ctypes.c_int32),
        ("srcs", ConvSrc * RSB_MAX_SRCS),
        ("nseg", ctypes.c_int32),
        ("segs", ConvSeg * RSB_MAX_SEGS),
        ("weights", ctypes.c_void_p),
        ("bias", ctypes.c_void_p),
        ("Cout", ctypes.c_int32),
        ("block_n", ctypes.c_int32),
        ("phases", ctypes.c_int32),
        ("Wt", ctypes.c_int32),
        ("Ht", ctypes.c_int32),
        ("Nt", ctypes.c_int32),
        ("TW", ctypes.c_int32),
        ("TH", ctypes.c_int32),
        ("TN", ctypes.c_int32),
        ("out", ctypes.c_void_p),
        ("out_pitch_w", ctypes.c_int64),
        ("out_pitch_h", ctypes.c_int64),
        ("out_pitch_n", ctypes.c_int64),
        ("out_sy", ctypes.c_int32),
        ("out_sx", ctypes.c_int32),
        ("residual", ctypes.c_void_p),
        ("relu", ctypes.c_int32),
        ("mode", ctypes.c_int32),
        ("head_classes", ctypes.c_int32),
        ("head_w", ctypes.c_void_p),
        ("head_b", ctypes.c_void_p),
        ("head_out", ctypes.c_void_p),
        ("cta_pair", ctypes.c_int32),
        ("split", ctypes.c_int32),
        ("out_plane", ctypes.c_int64),
        ("res_plane", ctypes.c_int64),
        ("acc_scale", ctypes.c_float),
        ("kchunk", ctypes.c_int32),
        ("scratch", ctypes.c_void_p),
        ("scratch_bytes", ctypes.c_int64),
        ("stats", ctypes.c_void_p),
        ("stats_bytes", ctypes.c_int64),
    ]


class RowConvDesc(ctypes.Structure):
    _fields_ = [
        ("src", ConvSrc),
        ("cin", ctypes.c_int32),
        ("taps_h", ctypes.c_int32),
        ("taps_w", ctypes.c_int32),
        ("dh0", ctypes.c_int32),
        ("dw0", ctypes.c_int32),
        ("nsub", ctypes.c_int32),
        ("nphase_a", ctypes.c_int32),
        ("weights", ctypes.c_void_p),
        ("bias", ctypes.c_void_p),
        ("Cout", ctypes.c_int32),
        ("Wt", ctypes.c_int32),
        ("Ht", ctypes.c_int32),
        ("Nt", ctypes.c_int32),
        ("out", ctypes.c_void_p),
        ("out_pitch_w", ctypes.c_int64),
        ("out_pitch_h", ctypes.c_int64),
        ("out_pitch_n", ctypes.c_int64),
        ("out_sy", ctypes.c_int32),
        ("out_sx", ctypes.c_int32),
        ("relu", ctypes.c_int32),
        ("mode", ctypes.c_int32),
        ("head_classes", ctypes.c_int32),
        ("head_w", ctypes.c_void_p),
        ("head_b", ctypes.c_void_p),
        ("head_out", ctypes.c_void_p),
        ("rows_per_unit", ctypes.c_int32),
        ("split", ctypes.c_int32),
        ("acc_scale", ctypes.c_float),
    ]


# name -> (restype, argtypes); mirrors include/rsb200.h one to one (tests/test_abi.py checks both sides)
_vp, _i32, _i64, _f32 = ctypes.c_void_p, ctypes.c_int32, ctypes.c_int64, ctypes.c_float
SIGNATURES = {
    "rsb_version": (ctypes.c_int, []),
    "rsb_abi_layout": (None, [ctypes.POINTER(_i32)]),
    "rsb_last_error": (ctypes.c_char_p, []),
    "rsb_device_ok": (ctypes.c_int, []),
    "rsb_conv_scratch_bytes": (_i64, [_i32]),
    "rsb_conv_plan_create": (ctypes.c_int, [ctypes.POINTER(ConvDesc), ctypes.POINTER(_vp)]),
    "rsb_conv_plan_destroy": (None, [_vp]),
    "rsb_conv_plan_info": (ctypes.c_int, [_vp] + [ctypes.POINTER(_i32)] * 4),
    "rsb_conv_run": (ctypes.c_int, [_vp, _vp]),
    "rsb_conv_run_simt_check": (ctypes.c_int, [ctypes.POINTER(ConvDesc), _vp]),
    "rsb_rowconv_plan_create": (ctypes.c_int, [ctypes.POINTER(RowConvDesc), ctypes.POINTER(_vp)]),
    "rsb_rowconv_plan_destroy": (None, [_vp]),
    "rsb_rowconv_run": (ctypes.c_int, [_vp, _vp]),
    "rsb_prepass_s2d": (ctypes.c_int, [_vp, _i32, _vp, _i32, _i32, _i32, ctypes.POINTER(_f32), ctypes.POINTER(_f32), _vp]),
    "rsb_prepass_s2d_split": (ctypes.c_int, [_vp, _i32, _vp, _i64, _i32, _i32, _i32, ctypes.POINTER(_f32), ctypes.POINTER(_f32), _vp]),
    "rsb_maxpool_nhwc": (ctypes.c_int, [_vp, _vp, _i32, _i32, _i32, _i32, _i32, _i32, _i32, _vp]),
    "rsb_maxpool_nhwc_split": (ctypes.c_int, [_vp, _i64, _vp, _i64, _i32, _i32, _i32, _i32, _i32, _i32, _i32, _vp]),
    "rsb_augment_dihedral": (ctypes.c_int, [_vp, _vp, _vp, _vp, _vp, _i32, _i32, _vp]),
    "rsb_head_quantize": (ctypes.c_int, [_vp, _vp, _vp, _i32, _i32, _i32, _i32, _vp]),
    "rsb_stitch_halo": (ctypes.c_int, [_vp, _vp, _vp, _i32, _i32, _i32, _vp]),
    "rsb_softvote": (ctypes.c_int, [_vp, _vp, _vp, _i32, _i64, _vp]),
    "rsb_class_histogram": (ctypes.c_int, [_vp, _i64, _i32, _vp, _vp]),
    "rsb_head_argmax": (ctypes.c_int, [_vp, _vp, _i32, _i32, _i32, _vp]),
    "rsb_zlib_inflate": (ctypes.c_int, [ctypes.c_char_p, _i64, _vp, _i64]),
    "rsb_png_decode_rgb": (ctypes.c_int, [_vp, _i64, _vp, _i32, _i32]),
    "rsb_png_read_rgb": (ctypes.c_int, [ctypes.c_char_p, _vp, _i32, _i32]),
    "rsb_png_encode_p8": (_i64, [_vp, _i32, _i32, _vp, _i32, _i32, _vp, _i64]),
    "rsb_png_write_p8": (ctypes.c_int, [ctypes.c_char_p, _vp, _i32, _i32, _vp, _i32, _i32]),
    "rsb_png_read_rgb_batch": (ctypes.c_int, [_vp, _i32, _vp, _i32, _i32, _i32, _vp]),
    "rsb_png_write_p8_batch": (ctypes.c_int, [_vp, _i32, _vp, _i64, _i32, _i32, _vp, _i32, _i32, _i32, _i32]),
    "rsb_softmax_nchw": (ctypes.c_int, [_vp, _vp, _i32, _i32, _i32, _vp]),
    "rsb_cross_entropy": (ctypes.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _i32, _vp]),
    "rsb_focal": (ctypes.c_int, [_vp, _vp, _vp, _f32, _vp, _vp, _vp, _i32, _i32, _i32, _vp]),
    "rsb_miou_scratch_doubles": (_i64, [_i32, _i32]),
    "rsb_miou": (ctypes.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _i32, _vp]),
    "rsb_lovasz_workspace_bytes": (_i64, [_i32, _i32, _i32]),
    "rsb_lovasz": (ctypes.c_int, [_vp, _vp, _vp, _vp, _vp, _i64, _i32, _i32, _i32, _vp]),
    "rsb_metrics_count": (ctypes.c_int, [_vp, _vp, _vp, _i32, _i32, _i32, _vp]),
    "rsb_adam_step": (ctypes.c_int, [_vp, _vp, _vp, _vp, _i64, _f32, _f32, _f32, _f32, _i32, _vp]),
    "rsb_adam_step_guarded": (ctypes.c_int, [_vp, _vp, _vp, _vp, _i64, _f32, _f32, _f32, _f32, _i32, _vp, _vp]),
    "rsb_bn_stats": (ctypes.c_int, [_vp, _vp, _i64, _i32, _vp]),
    "rsb_bn_stats_finalize": (ctypes.c_int, [_vp] * 11 + [_i64, _i32, _f32, _f32, _vp]),
    "rsb_bn_stats_finalize_chained": (ctypes.c_int, [_vp] * 11 + [_i64, _i32, _f32, _f32, _vp]),
    "rsb_bn_apply_chained": (ctypes.c_int, [_vp] * 5 + [_i64, _i32, _i32, _vp]),
    "rsb_bn_backward_chained": (ctypes.c_int, [_vp] * 13 + [_f32, _i64, _i32, _vp]),
    "rsb_bn_partials_finalize": (ctypes.c_int, [_vp, _i64] + [_vp] * 10 + [_i64, _i32, _f32, _f32, _i32, _vp]),
    "rsb_bn_finalize": (ctypes.c_int, [_vp] * 10 + [_i32, _i64, _f32, _f32, _vp]),
    "rsb_bn_apply": (ctypes.c_int, [_vp] * 5 + [_i64, _i32, _i32, _vp]),
    "rsb_bn_backward": (ctypes.c_int, [_vp] * 13 + [_f32, _i64, _i32, _vp]),
    "rsb_relu_backward": (ctypes.c_int, [_vp, _vp, _vp, _vp, _i64, _vp]),
    "rsb_multi_axpy": (ctypes.c_int, [_vp, _i32, ctypes.c_float, _vp]),
    "rsb_maxpool_backward": (ctypes.c_int, [_vp, _vp, _vp, _vp] + [_i32] * 7 + [_vp]),
    "rsb_final_forward": (ctypes.c_int, [_vp, _vp, _vp, _vp, _i32, _i32, _i32, _vp]),
    "rsb_final_backward": (ctypes.c_int, [_vp] * 7 + [_f32, _i32, _i32, _i32, _vp]),
    "rsb_pack_weights": (ctypes.c_int, [_vp, _vp, _vp, _i64, _vp]),
    "rsb_pack_weights1": (ctypes.c_int, [_vp, _vp, _vp, _i64, _vp]),
    "rsb_unpack_grads": (ctypes.c_int, [_vp, _vp, _vp, _i64, _f32, _vp]),
    "rsb_unpack_grads_gather": (ctypes.c_int, [_vp, _vp, _vp, _vp, _i64, _f32, _vp]),
    "rsb_pack_weights_split": (ctypes.c_int, [_vp, _vp, _vp, _i64, _i64, _f32, _vp, _vp]),
    "rsb_pack_weights1_split": (ctypes.c_int, [_vp, _vp, _vp, _i64, _i64, _f32, _vp, _vp]),
    "rsb_bn_stats_finalize_split": (ctypes.c_int, [_vp, _i64] + [_vp] * 10 + [_i64, _i32, _f32, _f32, _vp, _vp]),
    "rsb_bn_stats_finalize_split_chained": (ctypes.c_int, [_vp, _i64] + [_vp] * 10 + [_i64, _i32, _f32, _f32, _vp, _vp]),
    "rsb_bn_apply_split": (ctypes.c_int, [_vp, _i64, _vp, _vp, _vp, _i64, _vp, _i64, _i64, _i32, _i32, _vp]),
    "rsb_bn_apply_split_chained": (ctypes.c_int, [_vp, _i64, _vp, _vp, _vp, _i64, _vp, _i64, _i64, _i32, _i32, _vp]),
    "rsb_maxpool_backward_split": (ctypes.c_int, [_vp, _i64, _vp, _vp, _vp] + [_i32] * 7 + [_vp]),
    "rsb_final_forward_split": (ctypes.c_int, [_vp, _i64, _vp, _vp, _vp, _vp, _i32, _i32, _i32, _vp]),
    "rsb_wgrad_plan_create":(ctypes.c_int, [ctypes.POINTER(ConvDesc), _vp, _vp, ctypes.POINTER(_vp)]),
    "rsb_wgrad_plan_scratch_bytes": (_i64, [_vp]),
    "rsb_wgrad_plan_set_scratch": (ctypes.c_int, [_vp, _vp, _i64]),
    "rsb_wgrad_plan_destroy": (None, [_vp]),
    "rsb_wgrad_run": (ctypes.c_int, [_vp, _vp]),
}

DEBUG_SIGNATURES = {  # librsb200_debug.so (include/rsb200_debug.h): bring-up probes, used by scripts/ only
    "rsb_debug_umma": (ctypes.c_int, [_vp, _i32, _i32, _vp, _vp] + [_i32] * 8 + [_vp]),
    "rsb_debug_mma_rate": (ctypes.c_int, [_vp] + [_i32] * 5 + [_vp]),
}

_lib = None
_debug_lib = None


def load_debug():
    """the bring-up probe library (not part of the product): scripts/gpu_probe_umma.py, scripts/gpu_mma_rate.py"""
    global _debug_lib
    if _debug_lib is None:
        lib = ctypes.CDLL(os.path.join(_HERE, "librsb200_debug.so"))
        for name, (res, args) in DEBUG_SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype, fn.argtypes = res, args
        _debug_lib = lib
    return _debug_lib


def load():
    """Load librsb200.so once; raise RsbError (never fall back) if it is not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RsbError(
            "librsb200.so is not built ({}): run `python -c 'import __graft_entry__ as g; g.build()'` "
            "or `sh robosat_b200/csrc/build.sh`. There is no CPU fallback.".format(LIB_PATH)
        )
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError here means header and library disagree
        fn.restype = res
        fn.argtypes = args
    sizes = (ctypes.c_int32 * 4)()
    lib.rsb_abi_layout(sizes)
    mine = [ctypes.sizeof(ConvSrc), ctypes.sizeof(ConvSeg), ctypes.sizeof(ConvDesc), ctypes.sizeof(RowConvDesc)]
    if list(sizes) != mine:
        raise RsbError("struct layout mismatch between include/rsb200.h as compiled ({}) and robosat_b200/_lib.py ({}): rebuild the library".format(list(sizes), mine))
    _lib = lib
    return lib


RSB_E_UNSUPPORTED = -4


def last_error():
    return load().rsb_last_error().decode("utf-8", "replace")


def check(rc, what):
    if rc != 0:
        raise RsbError("{} failed (rc={}): {}".format(what, rc, last_error()))


def require_device():
    """Fail loudly unless a B200-class device and the TMA driver entry point are usable."""
    check(load().rsb_device_ok(), "rsb_device_ok")


def current_stream_ptr():
    import torch

    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
