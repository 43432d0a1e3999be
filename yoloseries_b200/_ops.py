"""Loader of the thin PyTorch C++ extension (csrc/torch_adapter.cpp -> _lib/libysb_torch.so, TORCH_LIBRARY namespace
``ysb``): the binding the hot entry points go through -- torch.ops.ysb.postprocess / filter_candidates / select_nms /
decode / decode_into / nms / pairwise_iou(_backward) / elementwise_iou(_backward) / match_tp / match_compact.

The extension checks tensors, picks torch's current stream on the tensors' device, allocates outputs from the caching
allocator and raises the reference's exception types; the arithmetic lives in libysb_postproc.so behind the C ABI
(include/ysb_postproc.h), which this module loads first (RTLD_GLOBAL) so that the extension's ysb_* symbols bind to it.
No fallback: a missing extension raises ImportError."""
import ctypes
import os

import torch

from . import _lib

ADAPTER_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "_lib", "libysb_torch.so")
_ops = None


def load():
    """Returns ``torch.ops.ysb`` (loads both shared libraries once)."""
    global _ops
    if _ops is None:
        _lib.load()
        if not os.path.exists(ADAPTER_PATH):
            raise ImportError(f"{ADAPTER_PATH} not found: build it with `python -m yoloseries_b200.build` "
                              "(or __graft_entry__.build()); yoloseries_b200 has no CPU/PyTorch fallback")
        torch.ops.load_library(ADAPTER_PATH)
        ops = torch.ops.ysb
        if ops.abi_version() != _lib.ABI_VERSION or ops.params_bytes() != ctypes.sizeof(_lib.YsbParams):
            raise ImportError("libysb_torch.so was built against another version of include/ysb_postproc.h")
        _ops = ops
    return _ops


def params_tensor(params):
    """CPU uint8 tensor sharing the memory of a ctypes YsbParams: what the extension's operators take as ``params``.
    Later writes to the struct's fields are seen by the operators."""
    return torch.frombuffer(params, dtype=torch.uint8)
