"""Python view of the module-level C entry points (``cmgan_tscnet_*`` in include/cmgan_b200.h): the same calls a C / C++ host makes.

``cmgan_tscnet_fwd`` runs TSCNet.forward (inference mode; ref: generator.py:174-196) from one flat parameter block and a caller-owned
workspace; torch is used here only to own the device memory."""
from __future__ import annotations

import ctypes
from typing import Dict, List, Tuple

import torch

from ._lib import lib


def param_table() -> List[Tuple[str, int, int]]:
    """[(state_dict key, offset in floats, element count)] of the flat parameter block, in state_dict order"""
    L = lib().cdll
    out = []
    key, off, n = ctypes.c_char_p(), ctypes.c_longlong(), ctypes.c_longlong()
    for i in range(L.cmgan_tscnet_param_count()):
        lib().call("cmgan_tscnet_param_info", i, ctypes.byref(key), ctypes.byref(off), ctypes.byref(n))
        out.append((key.value.decode(), off.value, n.value))
    return out


def pack_params(state_dict: Dict[str, torch.Tensor], device) -> torch.Tensor:
    """state_dict (reference key names) -> the flat fp32 block ``cmgan_tscnet_fwd`` reads"""
    flat = torch.zeros(lib().cdll.cmgan_tscnet_param_floats(), dtype=torch.float32, device=device)
    for key, off, n in param_table():
        t = state_dict[key]
        assert t.numel() == n, f"{key}: {t.numel()} elements, the C table expects {n}"
        flat[off:off + n].copy_(t.detach().reshape(-1).to(torch.float32))
    return flat


def workspace_bytes(B: int, T: int, F: int, precision: int) -> int:
    n = lib().cdll.cmgan_tscnet_workspace_bytes(B, T, F, precision)
    if n < 0:
        raise RuntimeError(lib().cdll.cmgan_last_error().decode())
    return n


def tscnet_forward(flat: torch.Tensor, x: torch.Tensor, precision: int = 1, workspace: torch.Tensor = None, frames: torch.Tensor = None):
    """x (B, 2, T, F) on the GPU, any strides -> (final_real, final_imag), each (B, 1, T, F).
    ``frames`` (optional, device int32 (B,)): ragged batch through ``cmgan_tscnet_fwd_varlen`` (frames t >= frames[b] unspecified)"""
    assert x.is_cuda and flat.is_cuda and x.dtype == torch.float32 and x.dim() == 4 and x.shape[1] == 2
    B, _, T, F = x.shape
    if workspace is None:
        workspace = torch.empty(workspace_bytes(B, T, F, precision), dtype=torch.uint8, device=x.device)
    fr = torch.empty(B, 1, T, F, device=x.device)
    fi = torch.empty(B, 1, T, F, device=x.device)
    sb, sc, st, sf = x.stride()
    if frames is not None:
        assert frames.is_cuda and frames.dtype == torch.int32 and frames.numel() == B and frames.is_contiguous()
        lib().call("cmgan_tscnet_fwd_varlen", flat.data_ptr(), x.data_ptr(), sb, sc, st, sf, B, T, F, frames.data_ptr(), fr.data_ptr(),
                   fi.data_ptr(), workspace.data_ptr(), workspace.numel(), precision, torch.cuda.current_stream().cuda_stream)
        return fr, fi
    lib().call("cmgan_tscnet_fwd", flat.data_ptr(), x.data_ptr(), sb, sc, st, sf, B, T, F, fr.data_ptr(), fi.data_ptr(), workspace.data_ptr(),
               workspace.numel(), precision, torch.cuda.current_stream().cuda_stream)
    return fr, fi
