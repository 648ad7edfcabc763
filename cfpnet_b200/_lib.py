"""ctypes binding of libcfp.so (the C ABI declared in include/cfp.h).

There is no fallback: if the library is missing or a call is rejected the
product path raises.  PyTorch is only the owner of device memory and streams;
every tensor is handed to the library as a raw device pointer.
"""
from __future__ import annotations

import ctypes as C
import os
import threading

import torch

from .geometry import ZoneGeometry

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("CFP_LIB_PATH") or os.path.join(_HERE, "libcfp.so")   # override: debug builds (tools/)

CFP_F32, CFP_BF16 = 0, 1
ABI_VERSION = 15
_fp = C.POINTER(C.c_float)


class CfpGeom(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        "zone_num", "pad_h", "pad_w", "p1", "p2", "sy_wo", "sx_wo", "ey_wo", "ex_wo",
        "tzh", "tzw", "interpolate", "ry0", "ry1", "rx0", "rx1")]

    @classmethod
    def from_geometry(cls, g: ZoneGeometry) -> "CfpGeom":
        return cls(**{n: getattr(g, n) for n, _ in cls._fields_})


class CfpLoftrW(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in (
        "wq_t", "wkv_t", "wm_t", "w1_t", "w2_t", "ln1_g", "ln1_b", "ln2_g", "ln2_b", "tc", "kv_tc")]


class CfpDapmW(C.Structure):
    _fields_ = [("attn", CfpLoftrW)] + [(n, C.c_void_p) for n in ("conv1_t", "shift1", "conv2_t", "shift2",
                                                                      "conv1_pk", "conv2_pk")]


class CfpLkpmW(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in (
        "dw_t", "dw_shift", "ln_g", "ln_b", "pw1_t", "pw1_b", "pw2_t", "pw2_b", "tc", "dw_toep")] + [("ksize", C.c_int32)]


class CfpTwinsW(C.Structure):
    _fields_ = [("lsa", CfpLoftrW), ("gsa", CfpLoftrW)] + \
               [(n, C.c_void_p) for n in ("sr_t", "sr_b", "srln_g", "srln_b", "sr_tc")] + [("ws", C.c_int32)]


class CfpHistW(C.Structure):
    _fields_ = [("w_t", C.c_void_p * 9), ("b", C.c_void_p * 9), ("tc", C.c_void_p)]


# name -> (restype, argtypes); must list every symbol include/cfp.h declares.
_i, _p, _sz, _i64 = C.c_int, C.c_void_p, C.c_size_t, C.c_int64
SIGNATURES = {
    "cfp_version": (_i, []),
    "cfp_last_error": (C.c_char_p, []),
    "cfp_workspace_bytes": (_sz, [_i, _i, _i, _i, _i, _i, _i, C.POINTER(CfpGeom)]),
    "cfp_geometry_from_rects": (_i, [_fp, _i, _i, _i, _i, _i, C.POINTER(CfpGeom)]),
    "cfp_hist_encoder_fwd": (_i, [_p, _p, _p, _p, _i64, C.POINTER(CfpHistW), _i, _p]),
    "cfp_zone_masks": (_i, [_p, _p, _p, _p, _i, _i, _i, C.POINTER(CfpGeom), _p]),
    "cfp_posenc_tokens_fwd": (_i, [_p, _p, _p, _i, _i, _i, _i, _i, _i, _i, _i, _i, _p]),
    "cfp_tokens_to_nchw": (_i, [_p, _p, _i, _i, _i, _i, _i, _p]),
    "cfp_d2i_fwd": (_i, [_p, _p, _p, _p, _p, _i, _i, _i, _i, _i, C.POINTER(CfpGeom),
                         C.POINTER(CfpLoftrW), _i, _p, _sz, _i, _p]),
    "cfp_dapm_fwd": (_i, [_p, _i, _i, _i, _i, C.POINTER(CfpGeom), C.POINTER(CfpDapmW), _p, _sz, _i, _p]),
    "cfp_lkpm_fwd": (_i, [_p, _i, _i, _i, _i, C.POINTER(CfpLkpmW), _p, _sz, _i, _p]),
    "cfp_twins_fwd": (_i, [_p, _i, _i, _i, _i, C.POINTER(CfpTwinsW), _p, _sz, _i, _p]),
    "cfp_twins_nchw_fwd": (_i, [_p, _p, _i, _i, _i, _i, C.POINTER(CfpTwinsW), _p, _sz, _i, _p]),
    "cfp_tr_gemm": (_i, [_p, _i64, _i64, _p, _i64, _i64, _p, _i64, _i, _i, _i, _p, _i, _p]),
    "cfp_tr_colsum": (_i, [_p, _p, _i64, _i, _p]),
    "cfp_tr_bn_stats": (_i, [_p, _i64, _i, C.c_float, C.c_float, _p, _p, _p, _p, _p, _p]),
    "cfp_tr_bn_apply": (_i, [_p, _p, _p, _p, _p, _p, _i64, _i, _i, _p]),
    "cfp_tr_bn_bwd": (_i, [_p, _p, _p, _p, _p, _p, _p, _p, _p, _i64, _i, _i, _p]),
    "cfp_tr_ln_fwd": (_i, [_p, _p, _p, _p, _i64, _i, C.c_float, _p]),
    "cfp_tr_ln_bwd": (_i, [_p, _p, _p, _p, _p, _p, _i64, _i, C.c_float, _p]),
    "cfp_tr_ew": (_i, [_p, _p, _p, _i64, _i, _p]),
    "cfp_tr_gather_rows": (_i, [_p, _p, _p, _i64, _i, _p]),
    "cfp_tr_scatter_add_rows": (_i, [_p, _p, _p, _p, _i64, _i64, _i, _p]),
    "cfp_tr_attn_reduce": (_i, [_p, _p, _p, _p, _p, _i, _i, _i, _i, _p]),
    "cfp_tr_attn_apply": (_i, [_p, _p, _p, _i, _i, _i, _i, _i, _p]),
    "cfp_tr_head_dot": (_i, [_p, _p, _p, _i64, _i, _i, _i, C.c_float, _p]),
    "cfp_tr_rowop": (_i, [_p, _p, _p, _p, _i64, _i, _i, _i, _i, _p]),
    "cfp_tr_dwconv": (_i, [_p, _p, _i, _i, _i, _i, _i, _p, _p, _i, _p]),
    "cfp_tr_dwconv_wgrad": (_i, [_p, _p, _p, _i, _i, _i, _i, _i, _p]),
    "cfp_tr_sumsq": (_i, [_p, _i64, C.c_float, _p, _p]),
    "cfp_tr_adamw": (_i, [_p, _p, _p, _p, _i64, _p, _p, _i] + [C.c_float] * 4 + [_i, C.c_float, _p, C.c_float, _p]),
    "cfp_conv_fwd": (_i, [_p] + [_i] * 7 + [_p, _p, C.c_float, _p, _i, _i, _p]),
    "cfp_upsample_concat": (_i, [_p, _i, _i, _i, _i, _p, _i, _p, _i, _i, _i, _i, _p]),
    "cfp_posenc_tokens_crop_fwd": (_i, [_p, _p, _p] + [_i] * 6 + [_p, _i, _p]),
    "cfp_posenc_tokens_nhwc_fwd": (_i, [_p, _i, _p, _p] + [_i] * 8 + [_p]),
    "cfp_copy_channels": (_i, [_p, _i, _p, _i, _i, _i, _i64, _p]),
    "cfp_head_bins": (_i, [_p, _i, _i, _i, _i] + [_p] * 7 + [_i, _i, C.c_float, C.c_float, _p, _p, _p, _p]),
    "cfp_head_expect": (_i, [_p, _i, _i, _i, _p, _p, _p, _i, _p, _p, _p]),
    "cfp_conv_f32_fwd": (_i, [_p] + [_i] * 6 + [_p, _p, C.c_float, _p, _i, _i, _p]),
    "cfp_upsample_concat_f32": (_i, [_p, _i, _i, _i, _i, _p, _i, _p, _i, _i, _i, _i, _p]),
    "cfp_posenc_tokens_nhwc_f32_fwd": (_i, [_p, _i, _p, _p] + [_i] * 8 + [_p]),
    "cfp_copy_channels_f32": (_i, [_p, _i, _p, _i, _i, _i, _i64, _p]),
    "cfp_head_bins_f32": (_i, [_p, _i, _i, _i, _i] + [_p] * 7 + [_i, _i, C.c_float, C.c_float, _p, _p, _p, _p]),
    "cfp_head_expect_f32": (_i, [_p, _i, _i, _i, _p, _p, _p, _i, _p, _p, _p]),
    "cfp_zone_hist": (_i, [_p] + [_i] * 9 + [C.c_float, _p, _p, _p, _p, _p]),
    "cfp_zone_samples": (_i, [_p, _p, _p, _i64, _i, _p, _p, _i, _p]),
    "cfp_silog_fwd": (_i, [_p, _p, _p] + [_i] * 6 + [_p, _p, _p]),
    "cfp_silog_bwd": (_i, [_p, _p, _p] + [_i] * 6 + [_p, C.c_float, _p, _p]),
    "cfp_depth_metrics": (_i, [_p, _p, _p, _i64, _p, _p, _p]),
    "cfp_launch_count": (_i64, []),
    "cfp_set_pdl": (_i, [_i]),
    "cfp_selftest_umma": (_i, [_p, _p, _p, _i, _i, _i, _i, _p]),
    "cfp_profile_start": (_i, []),
    "cfp_profile_stop": (_i, [C.c_char_p, _sz]),
}

_lib = None
_lock = threading.Lock()


class CfpError(RuntimeError):
    pass


def load() -> C.CDLL:
    """Load libcfp.so (once).  Raises CfpError when it has not been built."""
    global _lib
    if _lib is None:
        with _lock:
            if _lib is None:
                if not os.path.exists(LIB_PATH):
                    raise CfpError(f"{LIB_PATH} not found: build it with `python -m cfpnet_b200.build` "
                                   "(there is no CPU or PyTorch fallback for the fusion path)")
                lib = C.CDLL(LIB_PATH)
                for name, (res, args) in SIGNATURES.items():
                    fn = getattr(lib, name)
                    fn.restype, fn.argtypes = res, args
                if lib.cfp_version() != ABI_VERSION:
                    raise CfpError(f"libcfp ABI {lib.cfp_version()} != expected {ABI_VERSION}; rebuild")
                _lib = lib
    return _lib


def call(name: str, *args) -> None:
    lib = load()
    rc = getattr(lib, name)(*args)
    if rc != 0:
        raise CfpError(f"{name}: {lib.cfp_last_error().decode()}")


def dtype_code(dt: torch.dtype) -> int:
    if dt == torch.float32:
        return CFP_F32
    if dt == torch.bfloat16:
        return CFP_BF16
    raise CfpError(f"libcfp serves float32 and bfloat16 activations, not {dt}")


def require_cuda(t: torch.Tensor, what: str) -> None:
    if not t.is_cuda:
        raise CfpError(f"{what} must live on a CUDA device: the fusion path has no CPU implementation "
                       f"(got device {t.device})")


def ptr(t) -> int:
    return 0 if t is None else t.data_ptr()


def stream_ptr() -> int:
    return torch.cuda.current_stream().cuda_stream


def set_pdl(on) -> int:
    """Programmatic dependent launch for this thread's calls (True / False / None = default); returns the previous setting."""
    return int(load().cfp_set_pdl(-1 if on is None else int(bool(on))))


def launch_count() -> int:
    return int(load().cfp_launch_count())


def profile_start() -> None:
    call("cfp_profile_start")


def profile_stop() -> dict:
    """{kernel name: (launches, total ms)} of the calls made by this thread since profile_start()."""
    import json
    buf = C.create_string_buffer(1 << 16)
    call("cfp_profile_stop", buf, len(buf))
    return {k: (int(v[0]), float(v[1])) for k, v in json.loads(buf.value.decode()).items()}
