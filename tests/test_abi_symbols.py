"""CPU-side checks of the drop-in boundary: the C-ABI library builds/loads and exports every symbol that
include/hidvae_b200.h declares; argument validation that needs no GPU returns the documented status codes."""
import ctypes
import os
import re

import pytest

from helpers import ROOT, lib_mod

HEADER = os.path.join(ROOT, "include", "hidvae_b200.h")


def _declared_symbols():
    text = open(HEADER).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(hv_[a-z0-9_]+)\s*\(", text)))


def test_header_symbols_are_exported_and_bound(lib_mod):
    declared = _declared_symbols()
    assert "hv_rq_forward" in declared and "hv_rq_backward" in declared and len(declared) >= 11
    raw = ctypes.CDLL(lib_mod.LIB_PATH)
    for name in declared:
        assert hasattr(raw, name), f"{name} declared in include/hidvae_b200.h but not exported"
        assert name in lib_mod.SIGNATURES, f"{name} has no ctypes signature in hidvae_b200/_lib.py"
    assert sorted(lib_mod.SIGNATURES) == declared


def test_version_and_error_channel(lib_mod):
    assert lib_mod.version() >= 100
    # shape validation happens before any CUDA call
    st = lib_mod.lib.hv_rq_forward(None, -1, 32, None, 3, 256, 2, 0, 0.25, None, 0, 0, None, None, None, None, None, 0,
                                   None, 0, None)
    assert st == lib_mod.HV_ERR_BAD_SHAPE and "bad shape" in lib_mod.last_error()
    st = lib_mod.lib.hv_rq_forward(None, 8, 32, None, 3, 256, lib_mod.HV_MODE_GUMBEL_SOFTMAX, 1, 0.25, None, 0, 0, None,
                                   None, None, None, None, 0, None, 0, None)
    assert st == lib_mod.HV_ERR_UNSUPPORTED and "GUMBEL" in lib_mod.last_error()
    st = lib_mod.lib.hv_rq_backward(None, 8, 32, None, 9, 256, 2, 1, 0.25, None, 0, 0, None, 0, 0, None, 0, None, None,
                                    None, None, 0, None)
    assert st == lib_mod.HV_ERR_UNSUPPORTED
    assert lib_mod.lib.hv_rq_forward(None, 0, 32, None, 3, 256, 2, 0, 0.25, None, 0, 0, None, None, None, None, None, 0,
                                     None, 0, None) == lib_mod.HV_OK  # empty batch is a no-op


def test_workspace_sizes(lib_mod):
    ws = lib_mod.lib.hv_workspace_bytes
    # config 1/2/3/5: operand images + the swizzled fp32 copy the resident-codebook kernel gathers from
    assert ws(lib_mod.HV_OP_RQ_FORWARD, 0, 32, 256, 3) == 3 * 256 * (4 * 32 + 32) + 3 * 256 * 32 * 4
    assert ws(lib_mod.HV_OP_RQ_FORWARD, 0, 32, 512, 3) == 3 * 512 * (4 * 32 + 32)      # two images per level: images only
    assert ws(lib_mod.HV_OP_RQ_FORWARD, 0, 64, 4096, 4) == 4 * 4096 * (4 * 64 + 32)    # config 4
    assert ws(lib_mod.HV_OP_RQ_FORWARD, 0, 20, 256, 3) == 0                            # no tcgen05 instantiation
    assert ws(lib_mod.HV_OP_RQ_BACKWARD, 0, 32, 256, 3) == 0


def test_no_cpu_fallback(lib_mod):
    import torch
    from hidvae_b200 import ops
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        ops.rq_forward(torch.zeros(4, 32), torch.zeros(3, 256, 32))
    if not torch.cuda.is_available():
        with pytest.raises(lib_mod.HidvaeError):
            lib_mod.device_info()
