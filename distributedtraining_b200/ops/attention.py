"""Causal self-attention op (packed qkv layout).

CUDA path: hand-written tcgen05 kernel (csrc/sm100_attention.cu) when built; the PyTorch reference otherwise.
"""
from __future__ import annotations

import ctypes
import math


from . import _lib, reference as ref


def _kernel_ok(qkv, T, hd) -> bool:
    if not _lib.use_kernels(qkv):
        return False
    L = _lib.lib()
    return hasattr(L, "dtb_attention_fwd") and hd in (64, 128)


def attention_fwd(qkv, out, lse, B, T, H, hd, Hkv=None, drop=None, kv_len=None):
    """``kv_len`` (int32 [B], optional): per-sequence count of un-padded keys -- the HF ``attention_mask`` of a right-padded batch."""
    Hkv = Hkv or H
    if _kernel_ok(qkv, T, hd):
        from . import _drop_args, _tick
        rc = _lib.lib().dtb_attention_fwd(_lib.ptr(qkv), _lib.ptr(out), _lib.ptr(lse), B, T, H, Hkv, hd, qkv.stride(0),
                                          out.stride(0), ctypes.c_float(1.0 / math.sqrt(hd)), _lib.stream_ptr(),
                                          *_drop_args(drop), _lib.ptr(kv_len))
        if rc != 0:
            raise RuntimeError(f"attention_fwd kernel failed ({rc})")
        _tick()
        return out
    return ref.attention_fwd(qkv, out, lse, B, T, H, hd, Hkv, drop, kv_len)


def attention_bwd(dout, qkv, out, lse, dqkv, B, T, H, hd, Hkv=None, drop=None, dbias=None, kv_len=None):
    """``dbias`` (fp32 [qkv_dim], optional): += column sums of dqkv (the qkv bias gradient) -- folded into the single-block
    kernel's epilogue when it applies (128 % T == 0, MHA), a separate colsum pass otherwise."""
    Hkv = Hkv or H
    if _kernel_ok(qkv, T, hd) and hasattr(_lib.lib(), "dtb_attention_bwd"):
        from . import _drop_args, _tick, colsum
        import os
        fold = dbias is not None and 128 % T == 0 and H == Hkv and not os.environ.get("DTB200_ATTN_NO_SMALL")
        rc = _lib.lib().dtb_attention_bwd(_lib.ptr(dout), _lib.ptr(qkv), _lib.ptr(out), _lib.ptr(lse), _lib.ptr(dqkv), B, T,
                                          H, Hkv, hd, qkv.stride(0), out.stride(0), ctypes.c_float(1.0 / math.sqrt(hd)),
                                          _lib.stream_ptr(), *_drop_args(drop), _lib.ptr(dbias) if fold else None, _lib.ptr(kv_len))
        if rc != 0:
            raise RuntimeError(f"attention_bwd kernel failed ({rc})")
        _tick()
        if dbias is not None and not fold:
            colsum(dqkv, dbias)
        return dqkv
    ref.attention_bwd(dout, qkv, out, lse, dqkv, B, T, H, hd, Hkv, drop, kv_len)
    if dbias is not None:
        ref.colsum(dqkv, dbias)
    return dqkv
