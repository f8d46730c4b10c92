"""ctypes binding of libhidvae_b200.so (include/hidvae_b200.h).

There is no CPU fallback and no alternative backend: if the shared library has not been built the import of
this module raises, and every compute entry point raises `HidvaeError` when the library reports a failure.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import c_char_p, c_double, c_float, c_int, c_int64, c_size_t, c_uint64, c_void_p, POINTER

_PKG_ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))  # .../hid-vae_b200
LIB_NAME = "libhidvae_b200.so"
LIB_PATH = os.environ.get("HIDVAE_B200_LIB", os.path.join(_PKG_ROOT, LIB_NAME))

# hv_status_t
HV_OK, HV_ERR_BAD_SHAPE, HV_ERR_UNSUPPORTED, HV_ERR_MISALIGNED, HV_ERR_CUDA, HV_ERR_NULL, HV_ERR_WORKSPACE = range(7)
# hv_forward_mode_t (== QuantizeForwardMode values, modules/quantize.py:17-20)
HV_MODE_GUMBEL_SOFTMAX, HV_MODE_STE, HV_MODE_ROTATION_TRICK = 1, 2, 3
# hv_algo_t
HV_ALGO_AUTO, HV_ALGO_TCGEN05, HV_ALGO_SIMT, HV_ALGO_SIMT_DIFF, HV_ALGO_TCGEN05_PREPACKED = 0, 1, 2, 3, 4
# hv_op_t
HV_OP_RQ_FORWARD, HV_OP_RQ_BACKWARD = 0, 1

_STATUS_NAMES = {
    HV_ERR_BAD_SHAPE: "HV_ERR_BAD_SHAPE", HV_ERR_UNSUPPORTED: "HV_ERR_UNSUPPORTED",
    HV_ERR_MISALIGNED: "HV_ERR_MISALIGNED", HV_ERR_CUDA: "HV_ERR_CUDA", HV_ERR_NULL: "HV_ERR_NULL",
    HV_ERR_WORKSPACE: "HV_ERR_WORKSPACE",
}

# every symbol include/hidvae_b200.h declares: name -> (restype, argtypes)
SIGNATURES = {
    "hv_version": (c_int, []),
    "hv_last_error": (c_char_p, []),
    "hv_device_info": (c_int, [POINTER(c_int), POINTER(c_int), POINTER(c_int)]),
    "hv_workspace_bytes": (c_size_t, [c_int, c_int64, c_int, c_int, c_int]),
    "hv_rq_pack_codebooks": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_size_t, c_void_p]),
    "hv_rq_forward": (c_int, [c_void_p, c_int64, c_int, c_void_p, c_int, c_int, c_int, c_int, c_float,
                              c_void_p, c_int64, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                              c_int, c_void_p, c_size_t, c_void_p]),
    "hv_rq_backward": (c_int, [c_void_p, c_int64, c_int, c_void_p, c_int, c_int, c_int, c_int, c_float,
                               c_void_p, c_int64, c_int64, c_void_p, c_int64, c_int64, c_void_p, c_int64,
                               c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "hv_sort_workspace_bytes": (c_size_t, [c_int64]),
    "hv_kmeans_accumulate": (c_int, [c_void_p, c_int64, c_int, c_void_p, c_void_p, c_int, c_void_p, c_void_p,
                                     c_void_p, c_void_p, c_size_t, c_void_p]),
    "hv_kmeans_finalize": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "hv_uniq_forward": (c_int, [c_void_p, c_int64, c_int64, c_int64, c_int64, c_void_p, c_int, c_float,
                                c_void_p, c_void_p, c_size_t, c_void_p]),
    "hv_uniq_backward": (c_int, [c_void_p, c_int64, c_int64, c_int64, c_int64, c_void_p, c_int, c_float, c_float,
                                 c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "hv_semid_dedup_workspace_bytes": (c_size_t, [c_int64]),
    "hv_semid_dedup": (c_int, [c_void_p, c_int64, c_int64, c_int64, c_int64, c_int, c_void_p, c_void_p, c_int64, c_void_p,
                               c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "hv_gumbel_supported": (c_int, [c_int, c_int]),
    "hv_gumbel_uniforms": (c_int, [c_int64, c_int, c_uint64, c_uint64, c_void_p, c_void_p]),
    "hv_gumbel_forward": (c_int, [c_void_p, c_int64, c_int, c_void_p, c_int, c_float, c_float, c_void_p, c_uint64, c_uint64,
                                  c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "hv_gumbel_backward": (c_int, [c_void_p, c_int64, c_int, c_void_p, c_int, c_float, c_float, c_void_p, c_uint64, c_uint64,
                                   c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "hv_gumbel_uniforms_devrng": (c_int, [c_int64, c_int, c_void_p, c_void_p, c_void_p]),
    "hv_gumbel_forward_devrng": (c_int, [c_void_p, c_int64, c_int, c_void_p, c_int, c_float, c_float, c_void_p, c_void_p,
                                         c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "hv_gumbel_backward_devrng": (c_int, [c_void_p, c_int64, c_int, c_void_p, c_int, c_float, c_float, c_void_p, c_void_p,
                                          c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "hv_encoder_workspace_bytes": (c_size_t, [c_int, POINTER(c_int)]),
    "hv_encoder_pack_weights": (c_int, [POINTER(c_void_p), c_int, POINTER(c_int), c_void_p, c_size_t, c_void_p]),
    "hv_encoder_forward": (c_int, [c_void_p, c_int64, c_int, POINTER(c_int), c_void_p, c_size_t, c_int, c_int, c_void_p,
                                   c_void_p]),
    "hv_encoder_forward_f16": (c_int, [c_void_p, c_int64, c_int, POINTER(c_int), c_void_p, c_size_t, c_int, c_int, c_void_p,
                                       c_void_p]),
    "hv_tag_heads_workspace_bytes": (c_size_t, [c_int, c_int, c_int, POINTER(c_int), c_int, c_int64, POINTER(c_size_t)]),
    "hv_tag_heads_pack": (c_int, [POINTER(c_void_p), c_int, c_int, c_int, c_int, POINTER(c_int), c_int, c_void_p, c_size_t,
                                  c_void_p]),
    "hv_tag_heads_forward": (c_int, [c_void_p, c_int64, c_int64, c_int64, c_int, c_int, c_int, POINTER(c_int), c_int, c_void_p,
                                     c_size_t, c_void_p, c_int64, c_int64, c_void_p, c_int64, c_int64, POINTER(c_void_p),
                                     c_void_p, c_size_t, c_void_p]),
    "hv_peer_allreduce_chunks": (c_int, [c_int64]),
    "hv_peer_allreduce_set_timeout_ms": (None, [c_int64]),
    "hv_peer_allreduce_status": (c_int, [ctypes.c_uint32, POINTER(c_int), POINTER(c_int)]),
    "hv_peer_allreduce": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p]),
}


class HidvaeError(RuntimeError):
    """A call into libhidvae_b200.so returned a non-zero hv_status_t."""

    def __init__(self, status: int, message: str):
        super().__init__(f"{_STATUS_NAMES.get(status, status)}: {message}")
        self.status = status


def _load() -> ctypes.CDLL:
    if not os.path.isfile(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} not found: the CUDA extension is not built. Run `make -C {_PKG_ROOT}` "
            "(or `python -c 'import __graft_entry__ as g; g.build()'` at the repo root). "
            "hidvae_b200 has no CPU fallback.")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (restype, argtypes) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError here = header and library out of sync
        fn.restype = restype
        fn.argtypes = argtypes
    return lib


lib = _load()


def last_error() -> str:
    msg = lib.hv_last_error()
    return msg.decode("utf-8", "replace") if msg else ""


def check(status: int) -> None:
    if status != HV_OK:
        raise HidvaeError(status, last_error())


def version() -> int:
    return int(lib.hv_version())


def device_info():
    sm, major, minor = c_int(0), c_int(0), c_int(0)
    check(lib.hv_device_info(ctypes.byref(sm), ctypes.byref(major), ctypes.byref(minor)))
    return sm.value, major.value, minor.value
