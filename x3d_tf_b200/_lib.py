"""ctypes binding of the C ABI declared in `include/x3d_b200.h`.

There is deliberately no fallback: if the shared library is missing or a call fails, an
exception is raised (the product path never silently runs on the CPU or through PyTorch ops).
"""
from __future__ import annotations

import ctypes as C
import os
import threading

LIB_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "lib", "libx3d_b200.so")

X3D_F32, X3D_BF16 = 0, 1


class X3DLibError(RuntimeError):
    pass


class PwArgs(C.Structure):
    _fields_ = [("A", C.c_void_p), ("Wt", C.c_void_p), ("bias", C.c_void_p), ("R", C.c_void_p),
                ("se", C.c_void_p), ("D", C.c_void_p),
                ("M", C.c_int64), ("K", C.c_int32), ("Nc", C.c_int32), ("lda", C.c_int32),
                ("ldw", C.c_int32), ("ldr", C.c_int32), ("ldd", C.c_int32),
                ("rows_per_clip", C.c_int64),
                ("a_dtype", C.c_int32), ("d_dtype", C.c_int32), ("swish", C.c_int32),
                ("relu", C.c_int32),
                ("gather", C.c_int32), ("T", C.c_int32), ("Ho", C.c_int32), ("Wo", C.c_int32),
                ("Hi", C.c_int32), ("Wi", C.c_int32), ("stride", C.c_int32)]


class PwTcArgs(C.Structure):
    _fields_ = [("A", C.c_void_p), ("Wp", C.c_void_p), ("bias", C.c_void_p), ("R", C.c_void_p),
                ("se", C.c_void_p), ("D", C.c_void_p),
                ("M", C.c_int64), ("K", C.c_int32), ("Nc", C.c_int32), ("lda", C.c_int32),
                ("ldr", C.c_int32), ("ldd", C.c_int32), ("Kpad", C.c_int32), ("Npad", C.c_int32),
                ("rows_per_clip", C.c_int64), ("swish", C.c_int32), ("relu", C.c_int32),
                ("A2", C.c_void_p), ("a2_nt", C.c_int64), ("K2", C.c_int32), ("a2_stride", C.c_int32),
                ("a2_hi", C.c_int32), ("a2_wi", C.c_int32),
                ("colmean", C.c_void_p), ("store_d", C.c_int32), ("reserved", C.c_int32)]


class ClipDesc(C.Structure):
    _fields_ = [("H", C.c_int32), ("W", C.c_int32), ("rh", C.c_int32), ("rw", C.c_int32),
                ("y0", C.c_int32), ("x0", C.c_int32), ("flip", C.c_int32)]


class JpegFrame(C.Structure):
    _fields_ = [("seg_off", C.c_int64), ("coef_off", C.c_int64), ("plane_off", C.c_int64), ("out_off", C.c_int64),
                ("seg_len", C.c_int32), ("H", C.c_int32), ("W", C.c_int32), ("hs", C.c_int32), ("vs", C.c_int32),
                ("tables", C.c_int32), ("status", C.c_int32), ("reserved", C.c_int32)]


class JpegHuff(C.Structure):
    _fields_ = [("maxcode", C.c_int32 * 18), ("valoffset", C.c_int32 * 18), ("lookup", C.c_uint16 * 256),
                ("huffval", C.c_uint8 * 256)]


class JpegTables(C.Structure):
    _fields_ = [("dc", JpegHuff * 2), ("ac", JpegHuff * 2), ("q", (C.c_uint16 * 64) * 4),
                ("comp_q", C.c_int32 * 3), ("comp_dc", C.c_int32 * 3), ("comp_ac", C.c_int32 * 3),
                ("reserved", C.c_int32)]


class JpegInterval(C.Structure):
    _fields_ = [("off", C.c_int64), ("len", C.c_int32), ("frame", C.c_int32), ("mcu0", C.c_int32),
                ("nmcu", C.c_int32)]


class JpegEncFrame(C.Structure):
    _fields_ = [("in_off", C.c_int64), ("coef_off", C.c_int64), ("word_off", C.c_int64), ("word_cap", C.c_int64),
                ("H", C.c_int32), ("W", C.c_int32), ("hs", C.c_int32), ("vs", C.c_int32), ("tables", C.c_int32),
                ("reserved", C.c_int32)]


class JpegEncTables(C.Structure):
    _fields_ = [("q", (C.c_uint16 * 64) * 2), ("code", (C.c_uint16 * 256) * 4), ("size", (C.c_uint8 * 256) * 4)]


class JpegEncResult(C.Structure):
    _fields_ = [("bits", C.c_int64), ("out_off", C.c_int64), ("len", C.c_int64), ("status", C.c_int32),
                ("reserved", C.c_int32)]


X3D_JPEG_ISLOW, X3D_JPEG_IFAST = 0, 1
X3D_JPEG_OVERFLOW = 4

# name -> (restype, argtypes); must list every symbol include/x3d_b200.h declares.
SIGNATURES = {
    "x3d_version": (C.c_int, []),
    "x3d_last_error": (C.c_char_p, []),
    "x3d_crc32c": (C.c_uint32, [C.c_void_p, C.c_size_t, C.c_uint32]),
    "x3d_stem_fwd": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                               C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                               C.c_int, C.c_void_p]),
    "x3d_stem_tc_fwd": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int,
                                  C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "x3d_pw_fwd": (C.c_int, [C.POINTER(PwArgs), C.c_void_p]),
    "x3d_tf32_split": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "x3d_pw_tf32_fwd": (C.c_int, [C.c_void_p] * 4 + [C.c_int64] + [C.c_int] * 5 + [C.c_void_p, C.c_void_p]),
    "x3d_dw_partial_blocks": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]),
    "x3d_dw3x3x3_fwd": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                  C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                  C.c_int, C.c_int, C.c_void_p]),
    "x3d_dw3x3x3_act_fwd": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                      C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                      C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "x3d_dw_planar_partial_blocks": (C.c_int, [C.c_int] * 5),
    "x3d_dw_planar_lane_permille": (C.c_int, [C.c_int] * 5),
    "x3d_dw3x3x3_planar_fwd": (C.c_int, [C.c_void_p] * 4 + [C.c_int] * 9 + [C.c_void_p]),
    "x3d_se_mlp_fwd": (C.c_int, [C.c_void_p, C.c_int, C.c_float, C.c_void_p, C.c_void_p,
                                 C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                 C.c_void_p]),
    "x3d_avgpool_fwd": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int64, C.c_int, C.c_int,
                                  C.c_void_p]),
    "x3d_softmax_viewmean_fwd": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                           C.c_void_p]),
    "x3d_pw_tc_fwd": (C.c_int, [C.POINTER(PwTcArgs), C.c_void_p]),
    "x3d_pw_tc_sampler_supported": (C.c_int, [C.c_int] * 3),
    "x3d_gather_rows_fwd": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int,
                                      C.c_int, C.c_int, C.c_void_p]),
    "x3d_expand_dw_partial_blocks": (C.c_int, [C.c_int] * 6),
    "x3d_expand_dw_fwd": (C.c_int, [C.c_void_p] * 7 + [C.c_int] * 11 + [C.c_void_p]),
    "x3d_expand_dw2_partial_blocks": (C.c_int, [C.c_int] * 6),
    "x3d_expand_dw2_fwd": (C.c_int, [C.c_void_p] * 7 + [C.c_int] * 12 + [C.c_void_p]),
    # ---- training step
    "x3d_colreduce": (C.c_int, [C.c_void_p] * 5 + [C.c_int64, C.c_int, C.c_int64, C.c_void_p, C.c_int, C.c_void_p]),
    "x3d_bn_finalize": (C.c_int, [C.c_void_p, C.c_int64, C.c_int, C.c_float, C.c_float] + [C.c_void_p] * 6),
    "x3d_bn_apply_fwd": (C.c_int, [C.c_void_p] * 6 + [C.c_int64, C.c_int, C.c_int, C.c_void_p]),
    "x3d_bn_bwd_apply": (C.c_int, [C.c_void_p] * 8 + [C.c_int64, C.c_int, C.c_void_p]),
    "x3d_d2f": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_float, C.c_void_p]),
    "x3d_pw_wgrad": (C.c_int, [C.c_void_p] * 3 + [C.c_int64] + [C.c_int] * 10 + [C.c_void_p]),
    "x3d_dw_dgrad": (C.c_int, [C.c_void_p] * 3 + [C.c_int] * 8 + [C.c_void_p]),
    "x3d_dw_wgrad": (C.c_int, [C.c_void_p] * 3 + [C.c_int] * 8 + [C.c_void_p]),
    "x3d_stem_convs_fwd": (C.c_int, [C.c_void_p] * 3 + [C.c_int] * 5 + [C.c_void_p]),
    "x3d_stem_convs_wgrad": (C.c_int, [C.c_void_p] * 3 + [C.c_int] * 5 + [C.c_void_p]),
    "x3d_tconv_fwd": (C.c_int, [C.c_void_p] * 3 + [C.c_int, C.c_int, C.c_int64, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "x3d_tconv_wgrad": (C.c_int, [C.c_void_p] * 3 + [C.c_int, C.c_int, C.c_int64, C.c_int, C.c_int, C.c_void_p]),
    "x3d_scale_swish_fwd": (C.c_int, [C.c_void_p] * 3 + [C.c_int64, C.c_int, C.c_int64, C.c_void_p]),
    "x3d_scale_swish_bwd": (C.c_int, [C.c_void_p] * 5 + [C.c_int64, C.c_int, C.c_int64, C.c_void_p]),
    "x3d_ew": (C.c_int, [C.c_void_p] * 3 + [C.c_int64, C.c_int, C.c_void_p]),
    "x3d_pool_bwd": (C.c_int, [C.c_void_p] * 2 + [C.c_int64, C.c_int, C.c_int64, C.c_float, C.c_int, C.c_void_p]),
    "x3d_strided_add": (C.c_int, [C.c_void_p] * 2 + [C.c_int] * 7 + [C.c_void_p]),
    "x3d_dropout_mask": (C.c_int, [C.c_void_p, C.c_int64, C.c_float, C.c_uint64, C.c_void_p]),
    "x3d_softmax_xent": (C.c_int, [C.c_void_p] * 4 + [C.c_int, C.c_int, C.c_float, C.c_void_p]),
    "x3d_adam_step": (C.c_int, [C.c_void_p] * 5 + [C.c_int64, C.c_float, C.c_float, C.c_float, C.c_float, C.c_void_p]),
    "x3d_sgd_nesterov_step": (C.c_int, [C.c_void_p] * 4 + [C.c_int64, C.c_float, C.c_float, C.c_void_p]),
    # ---- either side of the path: input stage and evaluation metrics
    "x3d_normalize_u8": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.POINTER(C.c_float),
                                   C.POINTER(C.c_float), C.c_float, C.c_int, C.c_void_p]),
    "x3d_eval_views_u8": (C.c_int, [C.c_void_p, C.c_void_p] + [C.c_int] * 7 + [C.c_void_p]),
    "x3d_video_clips_u8": (C.c_int, [C.c_void_p] * 3 + [C.c_int] * 3 + [C.c_void_p, C.c_void_p]),
    "x3d_jpeg_entropy": (C.c_int, [C.c_void_p] * 3 + [C.c_int] + [C.c_void_p] * 3),
    "x3d_jpeg_entropy_rst": (C.c_int, [C.c_void_p] * 4 + [C.c_int] + [C.c_void_p] * 3),
    "x3d_jpeg_idct": (C.c_int, [C.c_void_p] * 3 + [C.c_int] * 3 + [C.c_void_p] * 2),
    "x3d_jpeg_color": (C.c_int, [C.c_void_p] * 2 + [C.c_int, C.c_int64] + [C.c_void_p] * 2),
    "x3d_jpeg_fdct": (C.c_int, [C.c_void_p] * 3 + [C.c_int] * 2 + [C.c_void_p] * 2),
    "x3d_jpeg_enc_bits": (C.c_int, [C.c_void_p] * 3 + [C.c_int] + [C.c_void_p] * 4),
    "x3d_jpeg_enc_emit": (C.c_int, [C.c_void_p] * 3 + [C.c_int] * 2 + [C.c_void_p] * 4),
    "x3d_jpeg_enc_stuff": (C.c_int, [C.c_void_p] * 2 + [C.c_int] + [C.c_void_p] * 2 + [C.c_int64, C.c_void_p]),
    "x3d_stem_tc_u8_fwd": (C.c_int, [C.c_void_p, C.POINTER(C.c_float), C.POINTER(C.c_float), C.c_float,
                                     C.c_void_p, C.c_void_p, C.c_void_p] + [C.c_int] * 6 + [C.c_void_p]),
    "x3d_eval_metrics": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                   C.c_void_p]),
    "x3d_head_fc_fwd": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int,
                                  C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
}

_lock = threading.Lock()
_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        with _lock:
            if _lib is None:
                if not os.path.exists(LIB_PATH):
                    raise X3DLibError(
                        f"{LIB_PATH} is missing: build it with `python -m x3d_tf_b200.build` "
                        "(nvcc, sm_100a).  There is no CPU or PyTorch fallback.")
                h = C.CDLL(LIB_PATH)
                for name, (res, args) in SIGNATURES.items():
                    fn = getattr(h, name)          # AttributeError if the symbol is not exported
                    fn.restype, fn.argtypes = res, args
                if h.x3d_version() != 100:
                    raise X3DLibError(f"ABI version mismatch: library reports {h.x3d_version()}")
                _lib = h
                try:
                    from . import tf_bundle
                    tf_bundle.set_native_crc32c(
                        lambda data, crc=0: h.x3d_crc32c(C.c_char_p(data), len(data), crc))
                except Exception:
                    pass
    return _lib


calls = 0          # C-ABI calls that returned a status (= kernel launches); bench.py reads the delta


def check(status: int, what: str = "") -> None:
    global calls
    calls += 1
    if status != 0:
        msg = lib().x3d_last_error().decode("utf-8", "replace")
        raise X3DLibError(f"{what or 'x3d call'} failed with status {status}: {msg}")
