"""Op layer: every hot op of the framework behind one functional API.

CUDA tensors are served by the hand-written sm_100a kernels in ``csrc/`` (through :mod:`._lib`); CPU tensors by the
PyTorch reference implementations in :mod:`.reference` (same signatures, used as test oracle).  There is no silent
fallback on a GPU box: if CUDA is available and the kernel library is missing the first call raises.
"""
from __future__ import annotations

import ctypes
import math
import os
from typing import Optional, Sequence

import torch

from . import _lib, reference as ref
from ._lib import have_kernels, use_kernels

EPI = {"none": 0, "bias": 1, "bias_gelu": 2, "bias_resid": 3, "dgelu": 4, "resid": 5}

_counters = {"launches": 0}


class DropoutRng:
    """Device-resident dropout state {seed, step counter}: masks are regenerated from it in forward AND backward
    (csrc/dropout.cuh); ``advance()`` is one tiny stream-ordered kernel, so a captured training step replays with fresh masks."""

    def __init__(self, device, seed: int = 0):
        self.state = torch.tensor([seed & 0x7FFFFFFF, 0, 0, 0], dtype=torch.int32, device=device)

    def advance(self) -> None:
        if use_kernels(self.state):
            _c(_lib.lib().dtb_rng_advance(_lib.ptr(self.state), _lib.stream_ptr()), "rng_advance")
            _tick()
        else:
            self.state[1] += 1


class Drop:
    """One dropout site: (rng state, site/stream id, probability)."""
    __slots__ = ("rng", "stream", "p")

    def __init__(self, rng: DropoutRng, stream: int, p: float):
        self.rng, self.stream, self.p = rng, int(stream), float(p)


def _drop_args(drop):
    if drop is None or drop.p <= 0.0:
        return None, 0, ctypes.c_float(0.0)
    return _lib.ptr(drop.rng.state), drop.stream, ctypes.c_float(drop.p)


def launch_count() -> int:
    """Number of hand-written kernel launches issued through this module (for bench.py's ``gpu_launches``)."""
    return _counters["launches"]


def _tick(n: int = 1) -> None:
    _counters["launches"] += n


def _c(rc: int, what: str) -> None:
    if rc != 0:
        raise RuntimeError(f"{what}: kernel launch failed (code {rc})")


def _row_major(t: torch.Tensor, what: str) -> int:
    assert t.dim() == 2 and t.stride(1) == 1, f"{what} must be a row-major 2D view"
    assert t.data_ptr() % 16 == 0, f"{what} must be 16-byte aligned"
    return t.stride(0)


# ---------------------------------------------------------------------------------------------------------------------
# GEMM
# ---------------------------------------------------------------------------------------------------------------------
def gemm(a, b, out, *, a_mn=False, b_mn=False, epi="none", bias=None, aux=None, out2=None, alpha=1.0, accumulate=False,
         splits=0, b2=None, b_persist=None, drop=None, colsum_out=None, ready=None):
    """out[M,N] = epi(alpha * A @ B^T) -- see :func:`reference.gemm` for the operand conventions.

    CUDA: persistent tcgen05/TMEM/TMA kernel (csrc/sm100_gemm.cu).  fp32 ``out`` is always reduce-ADDED by TMA
    (split-K capable); pass ``accumulate=False`` to have it zeroed first.

    ``b2``: second B operand of the same shape -- computes ``A (B + B2)^T`` as two accumulating tensor-core passes (the
    validator's ``theta_base + delta_i`` eval without materialising the sum; B2 may live in a peer window).
    ``b_persist``: local destination of the same shape as ``b`` -- when ``b`` is read from a PEER window (fused
    broadcast -> first forward GEMM) every B tile is also TMA-stored there while the MMA consumes it.
    ``drop`` (``Drop``, residual epilogues only): ``out = aux + dropout(alpha A B^T + bias)``, mask generated in the epilogue.
    ``colsum_out`` (fp32 [N], bf16 outputs): += column sums of ``out`` from the epilogue's staged tiles (a bias gradient that
    equals colsum of this GEMM's output, without a second pass over it).
    ``ready`` = (flags_address, target_tensor, hi): fused broadcast -> GEMM -- the kernel acquires flag slots 0..hi of this
    rank's base-flag block against the device-resident target round before touching ``b`` (the weights of a NEW averaged base
    that the shard owners' averaging kernels are landing in local HBM by multimem.st).
    """
    if not use_kernels(out):
        ref.gemm(a, b, out, a_mn=a_mn, b_mn=b_mn, epi=epi, bias=bias, aux=aux, out2=out2, alpha=alpha,
                 accumulate=accumulate, b2=b2, b_persist=b_persist, drop=drop)
        if colsum_out is not None:
            ref.colsum(out, colsum_out)
        return out
    assert a.dtype == torch.bfloat16 and b.dtype == torch.bfloat16
    lda, ldb, ldc = _row_major(a, "a"), _row_major(b, "b"), _row_major(out, "out")
    M, K = (a.shape[1], a.shape[0]) if a_mn else (a.shape[0], a.shape[1])
    N, Kb = (b.shape[1], b.shape[0]) if b_mn else (b.shape[0], b.shape[1])
    assert K == Kb, f"reduction dims differ: {K} vs {Kb}"
    assert out.shape[0] == M and out.shape[1] == N, f"out {tuple(out.shape)} != ({M},{N})"
    out_f32 = out.dtype == torch.float32
    if out_f32:
        assert epi == "none"
        if not accumulate:
            out.zero_()
        if splits <= 0:
            tiles = ((M + 127) // 128) * ((N + 255) // 256)
            nkb = (K + 63) // 64
            splits = max(1, min(nkb // 4 if nkb >= 8 else 1, (2 * _lib.num_sms()) // max(tiles, 1)))
    else:
        assert out.dtype == torch.bfloat16 and not accumulate
        splits = 1
    ldaux = _row_major(aux, "aux") if aux is not None else 0
    ldc2 = _row_major(out2, "out2") if out2 is not None else 0
    if ready is not None:
        _lib.lib().dtb_gemm_set_ready(ctypes.c_void_p(ready[0]), _lib.ptr(ready[1]), int(ready[2]))
    rc = _lib.lib().dtb_gemm_bf16(
        _lib.ptr(a), _lib.ptr(b), _lib.ptr(out), M, N, K, lda, ldb, ldc, int(a_mn), int(b_mn), int(out_f32), EPI[epi],
        _lib.ptr(bias), _lib.ptr(aux), ldaux, _lib.ptr(out2), ldc2, ctypes.c_float(alpha), splits, _lib.num_sms(),
        _lib.stream_ptr(), _lib.ptr(b2), _row_major(b2, "b2") if b2 is not None else 0, _lib.ptr(b_persist),
        _row_major(b_persist, "b_persist") if b_persist is not None else 0, *_drop_args(drop), _lib.ptr(colsum_out))
    _c(rc, "gemm")
    _tick()
    return out


class Fp8Scale:
    """Delayed per-tensor scaling state for one fp8 (e4m3) tensor: ``scale`` is used THIS step, ``amax`` is collected for
    the next one (``roll()`` once per step: scale <- max(amax, tiny) / 448, amax <- 0).  All on the device."""

    E4M3_MAX = 448.0

    def __init__(self, device, init_scale: float = 1.0 / 448.0 * 8.0):
        self.scale = torch.full((1,), init_scale, dtype=torch.float32, device=device)
        self.amax = torch.zeros(1, dtype=torch.float32, device=device)

    def roll(self) -> None:
        torch.maximum(self.amax, torch.full_like(self.amax, 1e-8), out=self.scale)
        self.scale.mul_(1.0 / self.E4M3_MAX)
        self.amax.zero_()


E5M2_MAX = 57344.0


def quantize_fp8(x, q, st: "Fp8Scale", e5m2: bool = False):
    """q (uint8 storage of e4m3, or e5m2 for gradients) = sat(x / st.scale); st.amax = max(st.amax, max|x|).  One pass."""
    if not use_kernels(x):
        st.amax.copy_(torch.maximum(st.amax, x.float().abs().max().reshape(1)))
        dt, mx = (torch.float8_e5m2, E5M2_MAX) if e5m2 else (torch.float8_e4m3fn, 448.0)
        q.view(dt).copy_((x.float() / st.scale).clamp(-mx, mx).to(dt))
        return q
    _c(_lib.lib().dtb_quant_fp8(_lib.ptr(x), _lib.ptr(q), _lib.ptr(st.scale), _lib.ptr(st.amax), ctypes.c_size_t(x.numel()),
                                _lib.num_sms(), _lib.stream_ptr(), int(e5m2)), "quant_fp8")
    _tick()
    return q


def quantize_fp8_t(w, q_t, st: "Fp8Scale"):
    """q_t [C, R] (e4m3) = sat(w [R, C] / st.scale)^T -- the transposed fp8 copy of a weight (K-major B operand of the fp8 dgrad)."""
    R, C = w.shape
    assert tuple(q_t.shape) == (C, R)
    if not use_kernels(w):
        q_t.view(torch.float8_e4m3fn).copy_((w.float() / st.scale).clamp(-448, 448).to(torch.float8_e4m3fn).t())
        return q_t
    _c(_lib.lib().dtb_quant_fp8_t(_lib.ptr(w), _lib.ptr(q_t), _lib.ptr(st.scale), R, C, _lib.stream_ptr()), "quant_fp8_t")
    _tick()
    return q_t


def gemm_fp8(a8, b8, out, sa: "Fp8Scale", sb: "Fp8Scale", *, epi="none", bias=None, aux=None, out2=None, drop=None,
             a_e5m2: bool = False):
    """out[M,N] (bf16) = epi(sa*sb * A8 @ B8^T) with fp8 operands (K-major), fp32 accumulation on kind::f8f6f4 tensor cores.
    A is e4m3 (forward activations) or, with ``a_e5m2``, e5m2 (activation gradients in the dgrad); B (a weight) is e4m3."""
    if not use_kernels(out):
        A = a8.view(torch.float8_e5m2 if a_e5m2 else torch.float8_e4m3fn).float() * sa.scale
        B = b8.view(torch.float8_e4m3fn).float() * sb.scale
        return ref.gemm(A, B, out, epi=epi, bias=bias, aux=aux, out2=out2, drop=drop)
    M, K = a8.shape
    N = b8.shape[0]
    assert b8.shape[1] == K and out.dtype == torch.bfloat16 and K % 16 == 0
    if a_e5m2:
        _lib.lib().dtb_gemm_fp8_a_e5m2()
    rc = _lib.lib().dtb_gemm_fp8(_lib.ptr(a8), _lib.ptr(b8), _lib.ptr(out), M, N, K, a8.stride(0), b8.stride(0), out.stride(0),
                                 EPI[epi], _lib.ptr(bias), _lib.ptr(aux), _row_major(aux, "aux") if aux is not None else 0,
                                 _lib.ptr(out2), _row_major(out2, "out2") if out2 is not None else 0, ctypes.c_float(1.0),
                                 _lib.num_sms(), _lib.stream_ptr(), _lib.ptr(sa.scale), _lib.ptr(sb.scale), *_drop_args(drop))
    _c(rc, "gemm_fp8")
    _tick()
    return out


# ---------------------------------------------------------------------------------------------------------------------
# embedding / norms / activations / loss
# ---------------------------------------------------------------------------------------------------------------------
def embed_fwd(ids, wte, wpe, out, wte2=None, wpe2=None, drop=None):
    """out = dropout(wte[ids] + wpe[pos] (+ wte2[ids] + wpe2[pos]: a second table, e.g. a delta in a peer window))."""
    if not use_kernels(out):
        if wte2 is not None:
            assert drop is None
            ref.embed_fwd(ids.long(), wte, wpe, out)
            tmp = torch.empty_like(out)
            ref.embed_fwd(ids.long(), wte2, wpe2, tmp)
            out.add_(tmp)
            return out
        return ref.embed_fwd(ids.long(), wte, wpe, out, drop)
    M, d = out.shape
    _c(_lib.lib().dtb_embed_fwd(_lib.ptr(ids), _lib.ptr(wte), _lib.ptr(wpe), _lib.ptr(out), M, ids.shape[-1], d,
                                _lib.stream_ptr(), _lib.ptr(wte2), _lib.ptr(wpe2), *_drop_args(drop)), "embed_fwd")
    _tick()
    return out


def embed_bwd(dx, ids, dwte, dwpe, drop=None):
    if not use_kernels(dx):
        return ref.embed_bwd(dx, ids.long(), dwte, dwpe, drop)
    M, d = dx.shape
    _c(_lib.lib().dtb_embed_bwd(_lib.ptr(dx), _lib.ptr(ids), _lib.ptr(dwte), _lib.ptr(dwpe), M, ids.shape[-1], d,
                                _lib.stream_ptr(), *_drop_args(drop)), "embed_bwd")
    _tick()


def layernorm_fwd(x, w, b, eps, out, mean, rstd):
    if not use_kernels(out):
        return ref.layernorm_fwd(x, w, b, eps, out, mean, rstd)
    M, d = x.shape
    _c(_lib.lib().dtb_norm_fwd(_lib.ptr(x), _lib.ptr(w), _lib.ptr(b), _lib.ptr(out), _lib.ptr(mean), _lib.ptr(rstd), M, d,
                               ctypes.c_float(eps), 0, _lib.stream_ptr()), "layernorm_fwd")
    _tick()
    return out


def layernorm_bwd(dy, x, w, mean, rstd, dx_out, dw, db, dresid=None, dcol=None, dxm=None, drop=None):
    """dx_out = LN'(dy) (+ dresid).  Two optional riders on the same pass:

    ``dxm`` + ``drop``: a second, dropout-masked copy of dx_out -- the dY of the GEMM whose output went through dropout
    site ``drop`` on its way into this residual stream (mask regenerated from the counter, never stored);
    ``dcol`` (fp32 [d]): += column sums of that dY (``dxm`` when given, else ``dx_out``) = the GEMM's bias gradient,
    instead of a separate colsum launch."""
    masked = dxm is not None and drop is not None and drop.p > 0
    if not use_kernels(dx_out):
        ref.layernorm_bwd(dy, x, w, mean, rstd, dx_out, dw, db, dresid)
        if masked:
            ref.masked_copy(dx_out, dxm, drop)
        if dcol is not None:
            ref.colsum(dxm if masked else dx_out, dcol)
        return dx_out
    M, d = x.shape
    fold = dcol is not None and d == 768
    _c(_lib.lib().dtb_norm_bwd(_lib.ptr(dy), _lib.ptr(x), _lib.ptr(w), _lib.ptr(mean), _lib.ptr(rstd), _lib.ptr(dresid),
                               _lib.ptr(dx_out), _lib.ptr(dw), _lib.ptr(db), M, d, 0, _lib.num_sms(), _lib.stream_ptr(),
                               _lib.ptr(dcol) if fold else None, _lib.ptr(dxm) if masked else None,
                               *_drop_args(drop if masked else None)), "layernorm_bwd")
    _tick()
    if dcol is not None and not fold:
        colsum(dxm if masked else dx_out, dcol)
    return dx_out


def rmsnorm_fwd(x, w, eps, out, rstd):
    if not use_kernels(out):
        return ref.rmsnorm_fwd(x, w, eps, out, rstd)
    M, d = x.shape
    _c(_lib.lib().dtb_norm_fwd(_lib.ptr(x), _lib.ptr(w), None, _lib.ptr(out), None, _lib.ptr(rstd), M, d,
                               ctypes.c_float(eps), 1, _lib.stream_ptr()), "rmsnorm_fwd")
    _tick()
    return out


def rmsnorm_bwd(dy, x, w, rstd, dx_out, dw, dresid=None):
    if not use_kernels(dx_out):
        return ref.rmsnorm_bwd(dy, x, w, rstd, dx_out, dw, dresid)
    M, d = x.shape
    _c(_lib.lib().dtb_norm_bwd(_lib.ptr(dy), _lib.ptr(x), _lib.ptr(w), None, _lib.ptr(rstd), _lib.ptr(dresid),
                               _lib.ptr(dx_out), _lib.ptr(dw), None, M, d, 1, _lib.num_sms(), _lib.stream_ptr(), None, None,
                               None, 0, ctypes.c_float(0.0)), "rmsnorm_bwd")
    _tick()
    return dx_out


def swiglu_fwd(gu, out):
    if not use_kernels(out):
        return ref.swiglu_fwd(gu, out)
    M, Fd = out.shape
    _c(_lib.lib().dtb_swiglu_fwd(_lib.ptr(gu), _lib.ptr(out), M, Fd, _lib.num_sms(), _lib.stream_ptr()), "swiglu_fwd")
    _tick()
    return out


def swiglu_bwd(dout, gu, dgu):
    if not use_kernels(dgu):
        return ref.swiglu_bwd(dout, gu, dgu)
    M, Fd = dout.shape
    _c(_lib.lib().dtb_swiglu_bwd(_lib.ptr(dout), _lib.ptr(gu), _lib.ptr(dgu), M, Fd, _lib.num_sms(), _lib.stream_ptr()),
       "swiglu_bwd")
    _tick()
    return dgu


def rope_(qkv, B, T, H, Hkv, hd, theta, inverse=False, inv_freq=None):
    """``inv_freq`` (fp32 [hd/2] on the device, optional): precomputed inverse frequencies (``models.transformer.rope_inv_freq``
    of a scaled config); None = ``theta ** (-2i/hd)`` computed inline."""
    if not use_kernels(qkv):
        return ref.rope_(qkv, B, T, H, Hkv, hd, theta, inverse, inv_freq)
    _c(_lib.lib().dtb_rope(_lib.ptr(qkv), B * T, T, H + Hkv, qkv.shape[1], hd, ctypes.c_float(theta), int(inverse),
                           _lib.num_sms(), _lib.stream_ptr(), _lib.ptr(inv_freq)), "rope")
    _tick()
    return qkv


def _qk_norm_kernel_ok(qkv, hd) -> bool:
    return use_kernels(qkv) and hd in (64, 128)


def qk_norm_rope_fwd(qkv, B, T, H, Hkv, hd, q_w, k_w, eps, inv_freq, raw=None, rstd=None):
    """Qwen3 QK-norm + RoPE, in place on the q|k part of packed qkv (see :func:`reference.qk_norm_rope_fwd`).
    ``inv_freq``: fp32 [hd/2] device table (``models.transformer.rope_inv_freq``).  ``raw`` / ``rstd``: optional saves for
    the backward.  CUDA: one warp per (row, q-or-k head), hd 64 and 128; other head dims take the reference path."""
    if not _qk_norm_kernel_ok(qkv, hd):
        return ref.qk_norm_rope_fwd(qkv, B, T, H, Hkv, hd, q_w, k_w, eps, inv_freq, raw, rstd)
    assert (raw is None) == (rstd is None)
    _c(_lib.lib().dtb_qk_norm_rope_fwd(_lib.ptr(qkv), _row_major(qkv, "qkv"), B * T, T, H, Hkv, hd, _lib.ptr(q_w),
                                       _lib.ptr(k_w), ctypes.c_float(eps), _lib.ptr(inv_freq), _lib.ptr(raw), _lib.ptr(rstd),
                                       _lib.num_sms(), _lib.stream_ptr()), "qk_norm_rope_fwd")
    _tick()
    return qkv


def qk_norm_rope_bwd(dqkv, B, T, H, Hkv, hd, q_w, k_w, inv_freq, raw, rstd, dq_w, dk_w):
    """Backward of :func:`qk_norm_rope_fwd`, in place on the q|k part of ``dqkv``; the norm-weight gradients ``dq_w`` /
    ``dk_w`` (fp32 [hd]) are accumulated."""
    if not _qk_norm_kernel_ok(dqkv, hd):
        return ref.qk_norm_rope_bwd(dqkv, B, T, H, Hkv, hd, q_w, k_w, inv_freq, raw, rstd, dq_w, dk_w)
    _c(_lib.lib().dtb_qk_norm_rope_bwd(_lib.ptr(dqkv), _row_major(dqkv, "dqkv"), B * T, T, H, Hkv, hd, _lib.ptr(q_w),
                                       _lib.ptr(k_w), _lib.ptr(inv_freq), _lib.ptr(raw), _lib.ptr(rstd), _lib.ptr(dq_w),
                                       _lib.ptr(dk_w), _lib.num_sms(), _lib.stream_ptr()), "qk_norm_rope_bwd")
    _tick()
    return dqkv


def ce_fwd_bwd(logits, targets, V, losses, grad_scale):
    if not use_kernels(logits):
        return ref.ce_fwd_bwd(logits, targets, V, losses, grad_scale)
    M, ldl = logits.shape[0], logits.stride(0)
    _c(_lib.lib().dtb_ce_fwd_bwd(_lib.ptr(logits), _lib.ptr(targets), _lib.ptr(losses), M, V, ldl,
                                 ctypes.c_float(grad_scale or 0.0), int(grad_scale is not None), _lib.stream_ptr()),
       "ce_fwd_bwd")
    _tick()
    return losses


_ATEN_SMALL = os.environ.get("DTB200_ATEN_SMALL", "0") == "1"  # A/B switch: ATen fill / sum instead of memset node / loss_mean_kernel


def loss_mean(losses, scale: float, out):
    """out[()] = scale * sum(losses): the step's mean loss in ONE deterministic launch (csrc/elementwise.cu loss_mean_kernel)."""
    if not use_kernels(losses) or _ATEN_SMALL:
        torch.sum(losses, dim=0, out=out)
        return out.mul_(scale)
    _c(_lib.lib().dtb_loss_mean(_lib.ptr(losses), losses.numel(), ctypes.c_float(scale), _lib.ptr(out), _lib.stream_ptr()), "loss_mean")
    _tick()
    return out


def zero_(t):
    """Stream-ordered memset (a memset node under graph capture) of a contiguous tensor."""
    if not use_kernels(t) or _ATEN_SMALL:
        return t.zero_()
    assert t.is_contiguous()
    _c(_lib.lib().dtb_zero(_lib.ptr(t), ctypes.c_size_t(t.numel() * t.element_size()), _lib.stream_ptr()), "zero")
    return t


def colsum(x, out):
    if not use_kernels(x):
        return ref.colsum(x, out)
    M, N = x.shape
    _c(_lib.lib().dtb_colsum(_lib.ptr(x), _lib.ptr(out), M, N, x.stride(0), _lib.stream_ptr()), "colsum")
    _tick()
    return out


# ---------------------------------------------------------------------------------------------------------------------
# attention
# ---------------------------------------------------------------------------------------------------------------------
def attention_fwd(qkv, out, lse, B, T, H, hd, Hkv=None, drop=None, kv_len=None):
    from . import attention as _att
    return _att.attention_fwd(qkv, out, lse, B, T, H, hd, Hkv, drop, kv_len)


def attention_bwd(dout, qkv, out, lse, dqkv, B, T, H, hd, Hkv=None, drop=None, dbias=None, kv_len=None):
    from . import attention as _att
    return _att.attention_bwd(dout, qkv, out, lse, dqkv, B, T, H, hd, Hkv, drop, dbias, kv_len)


# ---------------------------------------------------------------------------------------------------------------------
# optimizer / delta / averaging
# ---------------------------------------------------------------------------------------------------------------------
class AdamState:
    """Device-resident hyper-parameters + step counter so the optimizer step is CUDA-graph replayable."""

    def __init__(self, device, lr, beta1=0.9, beta2=0.999, eps=1e-6, weight_decay=0.0, grad_scale=1.0):
        self.device = torch.device(device)
        # [8] = "fresh": first step after (re-)creation -> the moments are implicitly zero (see csrc/optim_avg.cu adam_prep)
        self.hyper = torch.tensor([lr, beta1, beta2, eps, weight_decay, grad_scale, 1.0, 1.0, 0.0, 0.0, 0.0, 0.0],
                                  dtype=torch.float32, device=device)
        self.step = torch.zeros((), dtype=torch.int32, device=device)
        self.host = dict(lr=lr, beta1=beta1, beta2=beta2, eps=eps, weight_decay=weight_decay, grad_scale=grad_scale)
        self.host_step = 0

    def set_lr(self, lr: float) -> None:
        self.host["lr"] = lr
        self.hyper[0:1].fill_(lr)

    def reset(self) -> None:
        self.step.zero_()
        self.host_step = 0


def adamw_step(master, p16, grad, m, v, state: AdamState, base=None, delta=None, fresh_src=None):
    """One fused AdamW step over the whole arena; optionally also emits ``delta = master_new - base`` (fp32 or bf16).
    ``fresh_src``: on the FIRST step after an optimizer (re-)creation the parameters are read from there instead of from
    ``master`` (theta == theta_base right after a pull: the round then never writes the master arena)."""
    state.host_step += 1
    if not use_kernels(master):
        h = state.host
        state.step += 1
        if state.host_step == 1:  # first step after (re-)creation: moments are zero by definition (lazy optimizer reset)
            m.zero_()
            v.zero_()
            if fresh_src is not None and fresh_src.data_ptr() != master.data_ptr():
                master.copy_(fresh_src)
        ref.adamw_step(master, p16, grad, m, v, lr=h["lr"], beta1=h["beta1"], beta2=h["beta2"], eps=h["eps"],
                       weight_decay=h["weight_decay"], step=state.host_step, grad_scale=h["grad_scale"])
        if delta is not None:
            ref.delta_emit(master, base, delta)
        return master
    L = _lib.lib()
    _c(L.dtb_adam_prep(_lib.ptr(state.step), _lib.ptr(state.hyper), _lib.stream_ptr()), "adam_prep")
    mode = 0 if delta is None else (1 if delta.dtype == torch.float32 else 2)
    _c(L.dtb_adamw(_lib.ptr(master), _lib.ptr(p16), _lib.ptr(grad), _lib.ptr(m), _lib.ptr(v), _lib.ptr(state.hyper),
                   _lib.ptr(base), _lib.ptr(delta), mode, ctypes.c_size_t(master.numel()), _lib.num_sms(),
                   _lib.stream_ptr(), _lib.ptr(fresh_src)), "adamw")
    _tick(2)
    return master


DELTA_MODES = {torch.float32: 0, torch.bfloat16: 1, torch.uint8: 2, getattr(torch, "float8_e4m3fn", None): 2}


def delta_emit(master, base, out, scales=None, bad=None):
    """out = master - base in out's dtype; fp8 (uint8/float8_e4m3fn storage) is block-scaled: ``scales`` fp32[n/32].
    ``bad`` (int32[1], optional): set to 1 when the delta holds a NaN/Inf -- the NaN screen done at the source."""
    if not use_kernels(master):
        if bad is not None and not bool(torch.isfinite(master.float() - base.float()).all()):
            bad.fill_(1)
        if scales is not None:
            return ref_delta_emit_fp8(master, base, out, scales)
        return ref.delta_emit(master, base, out)
    mode = DELTA_MODES[out.dtype]
    _c(_lib.lib().dtb_delta_emit(_lib.ptr(master), _lib.ptr(base), _lib.ptr(out), _lib.ptr(scales),
                                 ctypes.c_size_t(master.numel()), mode, _lib.num_sms(), _lib.stream_ptr(), _lib.ptr(bad)),
       "delta_emit")
    _tick()
    return out


def ref_delta_emit_fp8(master, base, out, scales):
    d = (master.float() - base.float()).view(-1, 32)
    amax = d.abs().amax(dim=1)
    sc = torch.where(amax > 0, amax / 448.0, torch.ones_like(amax))
    q = (d / sc[:, None]).clamp(-448, 448).to(torch.float8_e4m3fn)
    out.view(torch.uint8).copy_(q.view(torch.uint8).reshape(-1))
    scales.copy_(sc)
    return out


def dequant_fp8(q, scales):
    return (q.view(torch.float8_e4m3fn).float().view(-1, 32) * scales[:, None]).reshape(-1)


def cast_copy(src, dst):
    if not use_kernels(src) or src.dtype != torch.float32 or dst.dtype != torch.bfloat16:
        return ref.cast_copy(src, dst)
    _c(_lib.lib().dtb_cast_f32_bf16(_lib.ptr(src), _lib.ptr(dst), ctypes.c_size_t(src.numel()), _lib.num_sms(),
                                    _lib.stream_ptr()), "cast")
    _tick()
    return dst


def round_reset(base, master, p16, m, v, reset_moments=True):
    """master = base, p16 = bf16(base), (m, v) = 0 in one pass (optimizer re-creation after a base pull)."""
    if not use_kernels(master):
        master.copy_(base)
        if p16 is not None and p16.data_ptr() != master.data_ptr():
            p16.copy_(base.to(p16.dtype))
        if reset_moments:
            m.zero_()
            v.zero_()
        return master
    _c(_lib.lib().dtb_round_reset(_lib.ptr(base), _lib.ptr(master), _lib.ptr(p16), _lib.ptr(m), _lib.ptr(v),
                                  ctypes.c_size_t(master.numel()), int(reset_moments), _lib.num_sms(), _lib.stream_ptr()),
       "round_reset")
    _tick()
    return master


def _ptr_array(ptrs: Sequence[int], ctype=ctypes.c_void_p):
    arr = (ctype * len(ptrs))()
    for i, p in enumerate(ptrs):
        arr[i] = p
    return arr


def _dp(t) -> int:
    """data pointer of a tensor, a raw int address (peer-mapped memory) or None."""
    if t is None:
        return 0
    return t if isinstance(t, int) else t.data_ptr()


def weighted_avg(base, deltas, w, manifest, outs_f32, outs_bf16=None, *, dscales=None, nan_flags=None, wait_flags=None,
                 wait_value=0, error_flag=None, chunk_range=None, mode=None, grid=None, chunk_ids=None, unit_base=False,
                 active=None, mc_f32: int = 0, mc_bf16: int = 0):
    """Fused kernel (a): ``theta_new = s_j*base + sum_i w[i,j]*delta_i`` written to every destination in ``outs_*``.

    ``deltas`` / ``outs_*`` entries are tensors or raw (peer-mapped) device addresses.  ``chunk_range`` restricts the
    launch to a shard of the manifest's chunk table (reduce-scatter form).  ``active`` (int32 [N], device): miners whose
    entry is 0 are neither read nor weighted (NaN / missing deltas, see :func:`round_prepare`).  ``mc_f32`` / ``mc_bf16``:
    MULTICAST addresses (parallel/symm.py ``SymmetricWindow.mc``): the result is additionally stored with ``multimem.st``, i.e.
    it lands in every rank's window -- the broadcast of the new base is part of the averaging kernel.  See csrc/optim_avg.cu.
    """
    N, P = w.shape
    if not isinstance(outs_f32, (list, tuple)):
        outs_f32 = [outs_f32]
    if outs_bf16 is not None and not isinstance(outs_bf16, (list, tuple)):
        outs_bf16 = [outs_bf16]
    if not use_kernels(base):
        tid = manifest.tensor_ids(base.device)
        dl = list(deltas)
        if dscales is not None:
            dl = [dequant_fp8(d, s) for d, s in zip(deltas, dscales)]
        if active is not None:
            keep = [i for i in range(N) if int(active[i]) != 0]
            dl, w = [dl[i] for i in keep], w[keep]
        tmp = torch.empty_like(base, dtype=torch.float32)
        ref.weighted_avg(base, dl, w, tid, tmp, nan_flags)
        if unit_base:
            tmp.add_(base * (1.0 - w.sum(0)[tid]))
        sel = None
        if chunk_ids is not None or chunk_range is not None:
            cs, cl, _ = manifest.seg_table(base.device)
            ids = chunk_ids if chunk_ids is not None else torch.arange(cs.numel())
            if chunk_range is not None:
                ids = ids[chunk_range[0]:chunk_range[1]]
            sel = torch.zeros(base.numel(), dtype=torch.bool, device=base.device)
            for c in ids.tolist():
                sel[int(cs[c]):int(cs[c]) + int(cl[c])] = True
        for o in list(outs_f32) + list(outs_bf16 or []):
            if o is not None:
                if sel is None:
                    o.copy_(tmp.to(o.dtype))
                else:
                    o[sel] = tmp[sel].to(o.dtype)
        return outs_f32[0] if outs_f32 else None
    cs, cl, ct = manifest.seg_table(base.device)
    c0, c1 = chunk_range if chunk_range is not None else (0, cs.numel() if chunk_ids is None else chunk_ids.numel())
    if mode is None:
        d0 = deltas[0]
        mode = 2 if dscales is not None else DELTA_MODES[d0.dtype]
    n_out = max(len(outs_f32), len(outs_bf16 or []))
    of = [_dp(o) for o in outs_f32] + [0] * (n_out - len(outs_f32))
    ob = [_dp(o) for o in (outs_bf16 or [])] + [0] * (n_out - len(outs_bf16 or []))
    rc = _lib.lib().dtb_gather_avg(
        _ptr_array([_dp(d) for d in deltas]), _ptr_array([_dp(s) for s in dscales]) if dscales is not None else None,
        _ptr_array([_dp(f) for f in wait_flags]) if wait_flags is not None else None, ctypes.c_uint32(wait_value),
        _lib.ptr(base), _lib.ptr(w), _lib.ptr(cs), _lib.ptr(cl), _lib.ptr(ct), c0, c1, _ptr_array(of), _ptr_array(ob),
        n_out, _lib.ptr(nan_flags), _lib.ptr(error_flag), N, P, mode, grid or _lib.num_sms() * 8, _lib.stream_ptr(),
        _lib.ptr(chunk_ids), int(unit_base), _lib.ptr(active), ctypes.c_void_p(mc_f32), ctypes.c_void_p(mc_bf16))
    _c(rc, "gather_avg")
    _tick()
    return outs_f32[0] if outs_f32 else None


def _first_chunk(manifest, device) -> torch.Tensor:
    """int32 [P + 1]: index of the first chunk of every manifest tensor in the chunk table."""
    key = ("first_chunk", str(device))
    cache = manifest._chunk_cache
    if key not in cache:
        _, _, ct = manifest.seg_table(device)
        first = torch.searchsorted(ct.long().contiguous(), torch.arange(len(manifest) + 1, device=device)).to(torch.int32)
        cache[key] = (first, first, first)
    return cache[key][0]


def seg_dot(gs, deltas, base, avg, manifest, dsts, *, N, gscales=None, wait_flags=None, wait_value=0, dscales=None, mode=0,
            chunk_range=None, active=None, loss=None, loss_scale=1.0, error_flag=None, partial=None):
    """Meta-gradient partial over a chunk range, for all miners at once (csrc/meta_avg.cu):

        dst[i*P + j] = sum_{e in tensor j, chunks [c0, c1)} gs[e] * (delta_i[e] + base[e] - avg[e]),   gs = sum_r gscales[r] * gs[r]

    ``gs`` / ``deltas`` / ``dsts`` entries are tensors or raw (peer-mapped) addresses; with R > 1 gradient arenas the
    reduce-scatter of the data-parallel validation gradients is fused into the dot.  ``dsts``: tables of N*P + 1 floats (the
    last entry receives ``loss * loss_scale``).  Deterministic (fixed reduction order)."""
    dev = base.device
    cs, cl, _ = manifest.seg_table(dev)
    P = len(manifest)
    c0, c1 = chunk_range if chunk_range is not None else (0, cs.numel())
    if partial is None:
        partial = torch.empty(max(c1 - c0, 1) * (N + 1), dtype=torch.float32, device=dev)
    R = len(gs)
    rc = _lib.lib().dtb_seg_dot(
        _ptr_array([_dp(g) for g in gs]), (ctypes.c_float * R)(*[float(x) for x in (gscales or [1.0] * R)]),
        _ptr_array([_dp(f) for f in wait_flags]) if wait_flags is not None else None, ctypes.c_uint32(wait_value), R,
        _ptr_array([_dp(d) for d in deltas]), _ptr_array([_dp(x) for x in dscales]) if dscales is not None else None, N, mode,
        _lib.ptr(base), _lib.ptr(avg), _lib.ptr(cs), _lib.ptr(cl), _lib.ptr(_first_chunk(manifest, dev)), c0, c1, P,
        _lib.ptr(partial), _ptr_array([_dp(d) for d in dsts]), len(dsts), _lib.ptr(active), _lib.ptr(loss),
        ctypes.c_float(loss_scale), _lib.ptr(error_flag), _lib.num_sms() * 4, _lib.stream_ptr())
    _c(rc, "seg_dot")
    _tick(2)


def multi_dot(g, deltas, base, avg, manifest, out, *, dscales=None, mode=None):
    """out[i,j] = <g_j, base_j + delta_ij - avg_j> for all miners i and manifest tensors j (segmented, one pass)."""
    N, P = out.shape
    if not use_kernels(g):
        tid = manifest.tensor_ids(g.device)
        dl = list(deltas)
        if dscales is not None:
            dl = [dequant_fp8(d, s) for d, s in zip(deltas, dscales)]
        return ref.multi_dot(g, dl, base, avg, tid, P, out)
    if mode is None:
        mode = 2 if dscales is not None else DELTA_MODES[deltas[0].dtype]
    table = torch.empty(N * P + 1, dtype=torch.float32, device=g.device)
    seg_dot([g], deltas, base, avg, manifest, [table], N=N, dscales=dscales, mode=mode)
    out.copy_(table[:N * P].view(N, P))
    return out


def round_prepare(delta_flags, bad_flags, round: int, active, n_active, w=None, init_w: bool = False, error_flag=None) -> None:
    """Start of an averaging round on the device (no host sync): wait for every miner's publish flag, read the NaN verdicts
    the miners attached to their publishes, write the ``active`` mask / count and optionally reset ``w`` to 1/n_active."""
    N = active.numel()
    P = w.shape[1] if w is not None else 0
    _c(_lib.lib().dtb_round_prepare(_ptr_array([_dp(f) for f in delta_flags]) if delta_flags is not None else None,
                                    _ptr_array([_dp(f) for f in bad_flags]) if bad_flags is not None else None,
                                    ctypes.c_uint32(round), _lib.ptr(active), _lib.ptr(n_active), _lib.ptr(w), N, P, int(init_w),
                                    _lib.ptr(error_flag), _lib.stream_ptr()), "round_prepare")
    _tick()


def shard_transpose(deltas, dscales, dsts, active, e0: int, e1: int, mode: int) -> None:
    """Delta all-to-all by pull: ``dsts[i][0 : e1-e0] = fp32(deltas[i][e0 : e1])`` for every miner i in one launch."""
    N = len(deltas)
    _c(_lib.lib().dtb_shard_transpose(_ptr_array([_dp(d) for d in deltas]),
                                      _ptr_array([_dp(x) for x in dscales]) if dscales is not None else None,
                                      _ptr_array([_dp(d) for d in dsts]), _lib.ptr(active), ctypes.c_size_t(e0), ctypes.c_size_t(e1),
                                      N, mode, _lib.num_sms() * 8, _lib.stream_ptr()), "shard_transpose")
    _tick()


def shard_pull16(srcs, manifest, chunks_per_rank: int, self_rank: int, dst, *, wait_flags=None, wait_value=0, error_flag=None) -> None:
    """bf16 all-gather by pull: every chunk NOT owned by ``self_rank`` is copied from its owner's (peer-mapped) buffer."""
    cs, cl, _ = manifest.seg_table(dst.device)
    _c(_lib.lib().dtb_shard_pull16(_ptr_array([_dp(x) for x in srcs]),
                                   _ptr_array([_dp(f) for f in wait_flags]) if wait_flags is not None else None,
                                   ctypes.c_uint32(wait_value), _lib.ptr(cs), _lib.ptr(cl), cs.numel(), chunks_per_rank, len(srcs),
                                   self_rank, _lib.ptr(dst), _lib.ptr(error_flag), _lib.num_sms() * 8, _lib.stream_ptr()),
       "shard_pull16")
    _tick()


def w_update(slots, w, lr: float, *, wait_flags=None, wait_value=0, loss_acc=None, error_flag=None) -> None:
    """``w -= lr * sum_r slots[r]`` (tables of N*P + 1 floats, summed in a fixed order); the loss shares go to ``loss_acc``."""
    N, P = w.shape
    _c(_lib.lib().dtb_w_update(_ptr_array([_dp(x) for x in slots]),
                               _ptr_array([_dp(f) for f in wait_flags]) if wait_flags is not None else None,
                               ctypes.c_uint32(wait_value), len(slots), _lib.ptr(w), ctypes.c_float(lr), N, P, _lib.ptr(loss_acc),
                               _lib.ptr(error_flag), _lib.stream_ptr()), "w_update")
    _tick()


def wait_flags_dev(flags_address: int, n: int, target: torch.Tensor, error_flag=None) -> None:
    """Stream-ordered device-side wait until flag slots 0..n-1 reach the round stored in ``target`` (device uint32/int32[1])."""
    _c(_lib.lib().dtb_wait_flags_dev(ctypes.c_void_p(flags_address), n, _lib.ptr(target), _lib.ptr(error_flag), _lib.stream_ptr()),
       "wait_flags_dev")
    _tick()


def set_flag_timeout(seconds: float) -> None:
    """Bound of every device-side flag spin (default ~13 s); <= 0 waits forever."""
    if have_kernels():
        L = _lib.lib()
        _c(L.dtb_set_flag_timeout_optim(ctypes.c_double(seconds)), "set_flag_timeout")
        _c(L.dtb_set_flag_timeout_meta(ctypes.c_double(seconds)), "set_flag_timeout")


def shard_pull_reset(shard_ptrs, manifest, chunks_per_rank, base_out, master, p16, m, v, *, reset_moments=True, wait_flags=None,
                     wait_value=0, error_flag=None):
    """All-gather-by-pull fused with the round reset: chunk c is read from ``shard_ptrs[c // chunks_per_rank]`` (peer-mapped
    base windows) and written to base_out / master / p16 (bf16) with the Adam moments cleared.  csrc/optim_avg.cu."""
    assert use_kernels(master), "shard_pull_reset is a peer-memory op (CUDA only)"
    cs, cl, _ = manifest.seg_table(master.device)
    world = len(shard_ptrs)
    rc = _lib.lib().dtb_shard_pull_reset(
        _ptr_array([_dp(x) for x in shard_ptrs]), _ptr_array([_dp(f) for f in wait_flags]) if wait_flags is not None else None,
        ctypes.c_uint32(wait_value), _lib.ptr(cs), _lib.ptr(cl), cs.numel(), chunks_per_rank, world, _lib.ptr(base_out),
        _lib.ptr(master), _lib.ptr(p16), _lib.ptr(m), _lib.ptr(v), int(reset_moments), _lib.ptr(error_flag),
        _lib.num_sms() * 8, _lib.stream_ptr())
    _c(rc, "shard_pull_reset")
    _tick()


def nvls_avg(delta_mc: int, out_mc: int, base: torch.Tensor, lo4: int, hi4: int, scale: float, base_scale: float = 1.0) -> None:
    """NVLS (in-switch) reduce + multicast broadcast of this rank's shard [lo4, hi4) (float4 units):
    ``out_all_ranks = base_scale * base + scale * sum_ranks(delta)``.  ``delta_mc`` / ``out_mc`` are multicast addresses
    of symmetric allocations (parallel.exchange.NvlsExchange); csrc/optim_avg.cu: nvls_avg_kernel."""
    assert use_kernels(base), "nvls_avg is an NVSwitch op (CUDA only)"
    assert base.numel() % 4 == 0 and base.dtype == torch.float32
    _c(_lib.lib().dtb_nvls_avg(ctypes.c_void_p(delta_mc), ctypes.c_void_p(out_mc), _lib.ptr(base), ctypes.c_size_t(lo4),
                               ctypes.c_size_t(hi4), ctypes.c_size_t(base.numel() // 4), ctypes.c_float(scale),
                               ctypes.c_float(base_scale), _lib.num_sms() * 8, _lib.stream_ptr()), "nvls_avg")
    _tick()


def checksum(flat: torch.Tensor) -> str:
    """Order-independent 128-bit device checksum of a flat fp32/bf16 arena (hex string).  CPU: same arithmetic in torch."""
    words = flat.contiguous().view(torch.int32)
    n = words.numel()
    if use_kernels(flat):
        out = torch.zeros(2, dtype=torch.int64, device=flat.device)
        _c(_lib.lib().dtb_checksum(_lib.ptr(words), ctypes.c_size_t(n), _lib.ptr(out), _lib.num_sms(), _lib.stream_ptr()), "checksum")
        _tick()
        a, b = [int(v) & 0xFFFFFFFFFFFFFFFF for v in out.tolist()]
    else:
        v = words.to(torch.int64) & 0xFFFFFFFF
        idx = (torch.arange(n, dtype=torch.int64) & 0xFFFFF) + 1
        a = int(v.sum().item()) & 0xFFFFFFFFFFFFFFFF
        b = 0
        for c0 in range(0, n, 1 << 20):  # python ints avoid int64 overflow of the weighted sum
            b = (b + int((v[c0:c0 + (1 << 20)] * idx[c0:c0 + (1 << 20)]).sum().item())) & 0xFFFFFFFFFFFFFFFF
    return f"{a:016x}{b:016x}"
