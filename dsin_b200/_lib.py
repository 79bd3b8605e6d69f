"""ctypes binding of libdsin_b200.so (the C ABI in include/dsin_b200.h).

There is no fallback: if the shared library is missing or the device is not sm_100,
importing the ops fails loudly (``DsinLibraryError``).
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libdsin_b200.so")


class DsinLibraryError(RuntimeError):
    pass


class ConvDesc(C.Structure):
    _fields_ = [(k, C.c_int) for k in
                ("n", "h", "w", "cin", "cout", "kh", "kw", "stride", "dilation", "transposed", "act", "post",
                 "dilation_x", "flags")]


ACT_NONE, ACT_RELU, ACT_LRELU02 = 0, 1, 2
POST_NONE, POST_DENORM_CLIP, POST_DENORM = 0, 1, 2

_P = C.c_void_p
_I = C.c_int
_I64 = C.c_int64

# name -> (restype, argtypes); must list every symbol declared in include/dsin_b200.h
SIGNATURES = {
    "dsin_version": (_I, []),
    "dsin_create": (_I, [C.POINTER(_P), _I]),
    "dsin_destroy": (_I, [_P]),
    "dsin_last_error": (C.c_char_p, [_P]),
    "dsin_launch_count": (_I64, [_P]),
    "dsin_nchw_to_nhwc": (_I, [_P, _P, _P, _I, _I, _I, _I, _I, _P]),
    "dsin_nhwc_to_nchw": (_I, [_P, _P, _P, _I, _I, _I, _I, _P]),
    "dsin_concat_normalize": (_I, [_P, _P, _P, _P, _I, _I, _I, _P]),
    "dsin_concat_normalize_split32": (_I, [_P, _P, _P, _P, _P, _I, _I, _I, _P]),
    "dsin_nchw_to_s2d_split32": (_I, [_P, _P, _P, _P, _I, _I, _I, _P]),
    "dsin_conv2d": (_I, [_P, C.POINTER(ConvDesc), _P, _P, _P, _P, _P, _P, _P, _P]),
    "dsin_pack_conv3x3_w": (_I, [_P, _P, _P, _P, _P, _I, _I, _P]),
    "dsin_conv3x3_c128_tc": (_I, [_P, _I, _I, _I, _P, _P, _P, _P, _P, _P, _I, _P, _P, _P, _P, _P, _P, _I, _P]),
    "dsin_conv_tc_npad": (_I, [_I]),
    "dsin_pack_conv_w_tc": (_I, [_P, _P, _I, _I, _I, _P, _P, _P, _P]),
    "dsin_conv2d_tc": (_I, [_P, C.POINTER(ConvDesc), _I] + [_P] * 14),
    "dsin_f32_to_split": (_I, [_P, _P, _P, _P, _I64, _P]),
    "dsin_split_to_f32": (_I, [_P, _P, _P, _P, _I64, _P]),
    "dsin_heatmap_quantize": (_I, [_P, _P, _P, _I, _I, _I, _I, _I, _P, _P, _P, _P, _P, _P, _P]),
    "dsin_probclass_workspace_bytes": (_I64, [_I, _I, _I, _I, _I]),
    "dsin_probclass_bits": (_I, [_P, _P, _P, _I, _I, _I, _I, _I, _I, C.c_float] + [_P] * 8 + [_P, _P, _P, _P]),
    "dsin_probclass_tc_workspace_bytes": (_I64, [_I, _I, _I, _I]),
    "dsin_probclass_bits_tc": (_I, [_P, _P, _P, _I, _I, _I, _I, C.c_float] + [_P] * 14 + [_I, _P, _P, _P, _P]),
    "dsin_sif_prepare": (_I, [_P, _P, _P, _I, _I, _I, _I, _I, _P, _P, _P, _P, _P]),
    "dsin_sif_workspace_bytes": (_I64, [_I, _I, _I, _I, _I, _I]),
    "dsin_sif_match": (_I, [_P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _P, _P, _P, _P, _P]),
    "dsin_sif_prepare_lab": (_I, [_P, _P, _P, _I, _I, _I, _I, _I, _P, _P, _P, _P, _P]),
    "dsin_sif_match_l2": (_I, [_P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _P, _P, _P, _P, _P]),
    "dsin_sif_work_count_offset": (_I64, [_P, _I, _I, _I, _I, _I]),
    "dsin_msssim_workspace_bytes": (_I64, [_I, _I, _I, _I, _I]),
    "dsin_msssim": (_I, [_P, _P, _P, _I, _I, _I, _I, _I, _P, _P, _P]),
    "dsin_validation_terms": (_I, [_P, _P, _P, _P, _P, _P, _I, _I64, _I64, _I, _P, _P]),
    "dsin_sif_gather": (_I, [_P, _P, _P, _P, _I, _I, _I, _I, _I, _P, _P]),
    "dsin_pc_codec_workspace_bytes": (_I64, [_I, _I, _I, _I]),
    "dsin_pc_encode": (_I, [_P, _P, _I, _I, _I, _I, _P, _I, _P, _I, _I, _P, _I64, _P, _P, _P, _P]),
    "dsin_pc_encode_wavefront": (_I, [_P, _P, _I, _I, _I, _I, _P, _I, _P, _I, _I, _P, _I64, _P, _P, _P, _P]),
    "dsin_pc_decode": (_I, [_P, _P, _I64, _P, _I, _I, _I, _I, _P, _I, _P, _I, _I, _P, _P, _P, _P]),
}

_lib = None


def load():
    """Load libdsin_b200.so and attach signatures.  Raises DsinLibraryError if absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise DsinLibraryError(
            "libdsin_b200.so not found at %s -- run `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a).  There is no CPU or PyTorch fallback." % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        try:
            fn = getattr(lib, name)
        except AttributeError:
            raise DsinLibraryError("libdsin_b200.so does not export %s (stale build?)" % name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


class Handle(object):
    """Owns one dsin_handle_t (one per device / per process)."""

    def __init__(self, device=0):
        self.lib = load()
        self._h = _P()
        rc = self.lib.dsin_create(C.byref(self._h), int(device))
        if rc != 0:
            raise DsinLibraryError(
                "dsin_create(device=%d) failed with code %d: libdsin_b200 needs an sm_100 (B200) GPU; "
                "there is no fallback path" % (device, rc))
        self.device = device

    def check(self, rc):
        if rc != 0:
            msg = self.lib.dsin_last_error(self._h)
            raise RuntimeError("libdsin_b200 error %d: %s" % (rc, msg.decode() if msg else "?"))

    @property
    def ptr(self):
        return self._h

    def launch_count(self):
        return int(self.lib.dsin_launch_count(self._h))

    def __del__(self):
        try:
            if self._h:
                self.lib.dsin_destroy(self._h)
                self._h = None
        except Exception:  # noqa: BLE001
            pass
