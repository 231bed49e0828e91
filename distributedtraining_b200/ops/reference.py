"""Plain-PyTorch reference implementation of every op in :mod:`distributedtraining_b200.ops`.

Used (a) on CPU (gloo plumbing tests, dev box), and (b) as the fp32 oracle the CUDA kernels are tested against.
All functions write into caller-provided output buffers so the engine code path is identical for both backends.
"""
from __future__ import annotations

import math
from typing import Sequence

import torch
import torch.nn.functional as F

GELU_K0 = math.sqrt(2.0 / math.pi)
GELU_K1 = 0.044715


# ---------------------------------------------------------------------------------------------------------------------
# counter-based dropout masks: the same arithmetic as csrc/dropout.cuh (uint32 math carried in int64)
# ---------------------------------------------------------------------------------------------------------------------
M32 = 0xFFFFFFFF


def _mix32s(x):
    x = (x * 0x7FEB352D) & M32
    x = x ^ (x >> 15)
    x = (x * 0x846CA68B) & M32
    return x ^ (x >> 16)


def _mix32(x):
    return _mix32s(x ^ (x >> 16))


def drop_thr(p: float) -> int:
    return int(p * 65536.0 + 0.5)


def drop_key(state, stream: int) -> int:
    """``state``: int32[4] tensor {seed, counter, -, -} (or a (seed, counter) tuple) -> the per-site 32-bit key."""
    seed, counter = (int(v) & M32 for v in (state[:2].tolist() if torch.is_tensor(state) else state[:2]))
    k = _mix32((seed + counter * 0x9E3779B9) & M32)
    return _mix32(k ^ ((stream * 0x85EBCA6B + 0xC2B2AE35) & M32))


def _bits16(word, odd):
    return torch.where(odd, word >> 16, word & 0xFFFF)


def drop_mult_2d(state, stream: int, p: float, M: int, d: int, device) -> torch.Tensor:
    """[M, d] fp32 multipliers (0 or 1/(1-p)) of a dropout site over a row-major [M, d] tensor."""
    key = drop_key(state, stream)
    r = torch.arange(M, dtype=torch.int64, device=device)[:, None]
    c = torch.arange(d, dtype=torch.int64, device=device)[None, :]
    pair = (r * (d >> 1) + (c >> 1)) & M32
    bits = _bits16(_mix32s(pair ^ key), (c & 1).bool())
    return (bits >= drop_thr(p)).float() * (1.0 / (1.0 - p))


def drop_mult_attn(state, stream: int, p: float, B: int, T: int, H: int, device) -> torch.Tensor:
    """[B, H, T, T] multipliers of the attention-probability dropout: element (b, h, i, j) is keyed by the q head, the
    global q row b*T + i and the global key token b*T + j."""
    key = drop_key(state, stream)
    M = B * T
    h = torch.arange(H, dtype=torch.int64, device=device)[None, :, None, None]
    b = torch.arange(B, dtype=torch.int64, device=device)[:, None, None, None]
    i = torch.arange(T, dtype=torch.int64, device=device)[None, None, :, None]
    j = torch.arange(T, dtype=torch.int64, device=device)[None, None, None, :]
    rowkey = _mix32((h * M + b * T + i) & M32 ^ key)
    kg = b * T + j
    bits = _bits16(_mix32s((kg >> 1) ^ rowkey), (kg & 1).bool())
    return (bits >= drop_thr(p)).float() * (1.0 / (1.0 - p))


def _drop_mult(drop, M, d, device):
    return None if drop is None or drop.p <= 0 else drop_mult_2d(drop.rng.state, drop.stream, drop.p, M, d, device)


def gelu_tanh(x: torch.Tensor) -> torch.Tensor:
    return F.gelu(x, approximate="tanh")


def dgelu_tanh(x: torch.Tensor) -> torch.Tensor:
    x2 = x * x
    u = GELU_K0 * (x + GELU_K1 * x * x2)
    t = torch.tanh(u)
    du = GELU_K0 * (1.0 + 3.0 * GELU_K1 * x2)
    return 0.5 * (1.0 + t) + 0.5 * x * (1.0 - t * t) * du


def gemm(a, b, out, *, a_mn=False, b_mn=False, epi="none", bias=None, aux=None, out2=None, alpha=1.0, accumulate=False,
         splits=1, b2=None, b_persist=None, drop=None):
    """out[M,N] = epi(alpha * A @ B^T).  ``a`` is stored [M,K] (K-major) or [K,M] (``a_mn``); ``b`` [N,K] or [K,N]."""
    A = a.t() if a_mn else a
    if b_persist is not None:
        b_persist.copy_(b)
    bb = b.float() + b2.float() if b2 is not None else b.float()
    Bt = bb if b_mn else bb.t()
    acc = (A.float() @ Bt) * alpha
    if epi in ("bias", "bias_gelu", "bias_resid"):
        acc = acc + bias.float()
    if epi == "bias_gelu":
        if out2 is not None:
            out2.copy_(acc.to(out2.dtype))
        acc = gelu_tanh(acc)
    elif epi in ("bias_resid", "resid"):
        mult = _drop_mult(drop, acc.shape[0], acc.shape[1], acc.device)
        if mult is not None:  # out = resid + dropout(A B^T + bias)
            acc = acc * mult
        acc = acc + aux.float()
    elif epi == "dgelu":
        acc = acc * dgelu_tanh(aux.float())
    elif epi != "none" and epi not in ("bias", "bias_gelu"):
        raise ValueError(f"unknown epilogue {epi!r}")
    if accumulate:
        out.add_(acc.to(out.dtype))
    else:
        out.copy_(acc.to(out.dtype))
    return out


def embed_fwd(ids, wte, wpe, out, drop=None):
    T = ids.shape[-1]
    x = wte[ids.reshape(-1)].float()
    if wpe is not None:
        pos = torch.arange(T, device=ids.device).repeat(ids.numel() // T)
        x = x + wpe[pos].float()
    mult = _drop_mult(drop, x.shape[0], x.shape[1], x.device)
    if mult is not None:
        x = x * mult
    out.copy_(x.to(out.dtype))
    return out


def embed_bwd(dx, ids, dwte, dwpe, drop=None):
    """dwte[V,d] += scatter(dx); dwpe[T,d] += sum over batch.  fp32 accumulators."""
    T = ids.shape[-1]
    d = dx.shape[-1]
    mult = _drop_mult(drop, dx.numel() // d, d, dx.device)
    if mult is not None:
        dx = dx.reshape(-1, d).float() * mult
    dwte.index_add_(0, ids.reshape(-1), dx.reshape(-1, d).to(dwte.dtype))
    if dwpe is not None:
        dwpe[:T].add_(dx.reshape(-1, T, d).to(dwpe.dtype).sum(0))


def layernorm_fwd(x, w, b, eps, out, mean, rstd):
    xf = x.float()
    mu = xf.mean(-1)
    var = xf.var(-1, unbiased=False)
    rs = torch.rsqrt(var + eps)
    y = (xf - mu[:, None]) * rs[:, None] * w.float() + b.float()
    out.copy_(y.to(out.dtype))
    mean.copy_(mu)
    rstd.copy_(rs)
    return out


def masked_copy(dx_out, dxm, drop):
    """dxm = dropout-masked copy of dx_out (the dY of the GEMM whose output went through dropout site ``drop``)."""
    mult = _drop_mult(drop, dx_out.shape[0], dx_out.shape[1], dx_out.device)
    dxm.copy_((dx_out.float() * mult).to(dxm.dtype))
    return dxm


def layernorm_bwd(dy, x, w, mean, rstd, dx_out, dw, db, dresid=None):
    """dx_out = LN'(dy) (+ dresid); dw/db (fp32) are ACCUMULATED."""
    dyf, xf = dy.float(), x.float()
    xhat = (xf - mean[:, None]) * rstd[:, None]
    dw.add_((dyf * xhat).sum(0))
    db.add_(dyf.sum(0))
    g = dyf * w.float()
    dx = (g - g.mean(-1, keepdim=True) - xhat * (g * xhat).mean(-1, keepdim=True)) * rstd[:, None]
    if dresid is not None:
        dx = dx + dresid.float()
    dx_out.copy_(dx.to(dx_out.dtype))
    return dx_out


def rmsnorm_fwd(x, w, eps, out, rstd):
    xf = x.float()
    rs = torch.rsqrt(xf.pow(2).mean(-1) + eps)
    out.copy_((xf * rs[:, None] * w.float()).to(out.dtype))
    rstd.copy_(rs)
    return out


def rmsnorm_bwd(dy, x, w, rstd, dx_out, dw, dresid=None):
    dyf, xf = dy.float(), x.float()
    xhat = xf * rstd[:, None]
    dw.add_((dyf * xhat).sum(0))
    g = dyf * w.float()
    dx = (g - xhat * (g * xhat).mean(-1, keepdim=True)) * rstd[:, None]
    if dresid is not None:
        dx = dx + dresid.float()
    dx_out.copy_(dx.to(dx_out.dtype))
    return dx_out


def _split_qkv(qkv, B, T, H, Hkv, hd):
    q, k, v = qkv.view(B, T, (H + 2 * Hkv) * hd).split([H * hd, Hkv * hd, Hkv * hd], dim=-1)
    q = q.view(B, T, H, hd).transpose(1, 2)
    k = k.view(B, T, Hkv, hd).transpose(1, 2)
    v = v.view(B, T, Hkv, hd).transpose(1, 2)
    return q, k, v


def attn_mask(B, T, device, kv_len=None):
    """[B,1,T,T] bool: key c is visible to query r iff c <= r (causal) and c < kv_len[b] (padding mask of a right-padded
    batch, HF ``attention_mask`` semantics: reference hivetrain/training_manager.py:380-384); kv_len is clamped to >= 1."""
    mask = torch.ones(T, T, dtype=torch.bool, device=device).tril()[None, None]
    if kv_len is not None:
        key_ok = torch.arange(T, device=device)[None, :] < kv_len.to(device).long().clamp(min=1)[:, None]
        mask = mask & key_ok[:, None, None, :]
    return mask.expand(B, 1, T, T)


def attention_fwd(qkv, out, lse, B, T, H, hd, Hkv=None, drop=None, kv_len=None):
    """Causal self-attention over packed qkv [B*T, (H+2Hkv)*hd] -> out [B*T, H*hd]; lse [B,H,T] fp32 (natural log).
    ``drop``: dropout on the softmax probabilities (the normaliser / lse are those of the un-dropped softmax)."""
    Hkv = Hkv or H
    q, k, v = _split_qkv(qkv, B, T, H, Hkv, hd)
    if Hkv != H:
        k = k.repeat_interleave(H // Hkv, dim=1)
        v = v.repeat_interleave(H // Hkv, dim=1)
    s = (q.float() @ k.float().transpose(-1, -2)) / math.sqrt(hd)
    mask = attn_mask(B, T, qkv.device, kv_len)
    s = s.masked_fill(~mask, float("-inf"))
    l = torch.logsumexp(s, dim=-1)
    p = torch.exp(s - l[..., None])
    if drop is not None and drop.p > 0:
        p = p * drop_mult_attn(drop.rng.state, drop.stream, drop.p, B, T, H, qkv.device)
    o = p @ v.float()
    out.copy_(o.transpose(1, 2).reshape(B * T, H * hd).to(out.dtype))
    if lse is not None:
        lse.copy_(l)
    return out


def attention_bwd(dout, qkv, out, lse, dqkv, B, T, H, hd, Hkv=None, drop=None, kv_len=None):
    Hkv = Hkv or H
    rep = H // Hkv
    q, k, v = _split_qkv(qkv, B, T, H, Hkv, hd)
    q, k, v = q.float(), k.float(), v.float()
    kx = k.repeat_interleave(rep, dim=1) if rep > 1 else k
    vx = v.repeat_interleave(rep, dim=1) if rep > 1 else v
    do = dout.view(B, T, H, hd).transpose(1, 2).float()
    o = out.view(B, T, H, hd).transpose(1, 2).float()
    scale = 1.0 / math.sqrt(hd)
    s = (q @ kx.transpose(-1, -2)) * scale
    mask = attn_mask(B, T, qkv.device, kv_len)
    p = torch.exp(s - lse[..., None]).masked_fill(~mask, 0.0)
    dp = do @ vx.transpose(-1, -2)
    if drop is not None and drop.p > 0:
        mult = drop_mult_attn(drop.rng.state, drop.stream, drop.p, B, T, H, qkv.device)
        dv = (p * mult).transpose(-1, -2) @ do
        dp = dp * mult
    else:
        dv = p.transpose(-1, -2) @ do
    D = (do * o).sum(-1, keepdim=True)
    ds = p * (dp - D) * scale
    dq = ds @ kx
    dk = ds.transpose(-1, -2) @ q
    if rep > 1:
        dk = dk.view(B, Hkv, rep, T, hd).sum(2)
        dv = dv.view(B, Hkv, rep, T, hd).sum(2)
    dq = dq.transpose(1, 2).reshape(B * T, H * hd)
    dk = dk.transpose(1, 2).reshape(B * T, Hkv * hd)
    dv = dv.transpose(1, 2).reshape(B * T, Hkv * hd)
    dqkv.copy_(torch.cat([dq, dk, dv], dim=-1).to(dqkv.dtype))
    return dqkv


def rope_(qkv, B, T, H, Hkv, hd, theta, inverse=False, inv_freq=None):
    """In-place rotary embedding (rotate-half convention) on the q and k parts of packed qkv.  ``inv_freq`` (fp32 [hd/2],
    optional) replaces the unscaled ``theta ** (-2i/hd)`` frequencies (see ``models.transformer.rope_inv_freq``)."""
    dev = qkv.device
    half = hd // 2
    if inv_freq is not None:
        inv = inv_freq.to(device=dev, dtype=torch.float32)
    else:
        inv = 1.0 / (theta ** (torch.arange(0, half, device=dev, dtype=torch.float32) / half))
    ang = torch.arange(T, device=dev, dtype=torch.float32)[:, None] * inv[None, :]
    cos, sin = ang.cos(), ang.sin()
    if inverse:
        sin = -sin
    x = qkv.view(B, T, H + 2 * Hkv, hd)
    qk = x[:, :, :H + Hkv].float()
    x1, x2 = qk[..., :half], qk[..., half:]
    c, s = cos[None, :, None, :], sin[None, :, None, :]
    r = torch.cat([x1 * c - x2 * s, x2 * c + x1 * s], dim=-1)
    x[:, :, :H + Hkv].copy_(r.to(qkv.dtype))
    return qkv


def _qk_norm_weights(q_w, k_w, H, Hkv):
    """[H + Hkv, hd] fp32: q_norm for the q heads, k_norm for the k heads."""
    return torch.cat([q_w.float()[None].expand(H, -1), k_w.float()[None].expand(Hkv, -1)])


def _rotate(x, T, inv, sign):  # x [B, T, h, hd] fp32, rotate-half by sign * t * inv
    half = x.shape[-1] // 2
    ang = torch.arange(T, device=x.device, dtype=torch.float32)[:, None] * inv.to(device=x.device, dtype=torch.float32)[None, :]
    c, s = ang.cos()[None, :, None, :], sign * ang.sin()[None, :, None, :]
    x1, x2 = x[..., :half], x[..., half:]
    return torch.cat([x1 * c - x2 * s, x2 * c + x1 * s], dim=-1)


def qk_norm_rope_fwd(qkv, B, T, H, Hkv, hd, q_w, k_w, eps, inv_freq, raw=None, rstd=None):
    """In place on the q|k part of packed qkv [B*T, (H+2Hkv)*hd]: per-head RMSNorm (``q_w`` for q heads, ``k_w`` for k heads,
    fp32 statistics) followed by rotate-half RoPE with the ``inv_freq`` table [hd/2].  v is not touched.  Optional saves
    for the backward: ``raw`` [B*T, (H+Hkv)*hd] = the q|k input, ``rstd`` [B*T, H+Hkv] fp32."""
    nh = H + Hkv
    x = qkv.view(B, T, H + 2 * Hkv, hd)
    qk = x[:, :, :nh].float()
    if raw is not None:
        raw.copy_(x[:, :, :nh].reshape(B * T, nh * hd))
    rs = torch.rsqrt(qk.pow(2).mean(-1) + eps)
    if rstd is not None:
        rstd.copy_(rs.reshape(B * T, nh))
    y = qk * rs[..., None] * _qk_norm_weights(q_w, k_w, H, Hkv)
    x[:, :, :nh].copy_(_rotate(y, T, inv_freq, 1.0).to(qkv.dtype))
    return qkv


def qk_norm_rope_bwd(dqkv, B, T, H, Hkv, hd, q_w, k_w, inv_freq, raw, rstd, dq_w, dk_w):
    """Backward of :func:`qk_norm_rope_fwd`, in place on the q|k part of dqkv: g = R(-theta) dy, x^ = raw * rstd,
    dx = rstd * (g w - x^ mean(g w x^)); ``dq_w`` / ``dk_w`` (fp32 [hd]) += sum of g x^ over rows and q / k heads."""
    nh = H + Hkv
    d = dqkv.view(B, T, H + 2 * Hkv, hd)
    g = _rotate(d[:, :, :nh].float(), T, inv_freq, -1.0)
    rs = rstd.view(B, T, nh, 1).float()
    xh = raw.view(B, T, nh, hd).float() * rs
    gw = g * _qk_norm_weights(q_w, k_w, H, Hkv)
    dx = rs * (gw - xh * (gw * xh).mean(-1, keepdim=True))
    gx = g * xh
    dq_w.add_(gx[:, :, :H].sum((0, 1, 2)).to(dq_w.dtype))
    dk_w.add_(gx[:, :, H:].sum((0, 1, 2)).to(dk_w.dtype))
    d[:, :, :nh].copy_(dx.to(dqkv.dtype))
    return dqkv


def swiglu_fwd(gu, out):
    """gu [M, 2F] = [gate | up] -> out [M,F] = silu(gate) * up."""
    Fdim = gu.shape[-1] // 2
    g, u = gu[:, :Fdim].float(), gu[:, Fdim:].float()
    out.copy_((F.silu(g) * u).to(out.dtype))
    return out


def swiglu_bwd(dout, gu, dgu):
    Fdim = gu.shape[-1] // 2
    g, u = gu[:, :Fdim].float(), gu[:, Fdim:].float()
    d = dout.float()
    sg = torch.sigmoid(g)
    dgu[:, :Fdim].copy_((d * u * sg * (1 + g * (1 - sg))).to(dgu.dtype))
    dgu[:, Fdim:].copy_((d * g * sg).to(dgu.dtype))
    return dgu


def ce_fwd_bwd(logits, targets, V, losses, grad_scale):
    """Row-wise CE over the first V columns of ``logits`` [M, ldl]; logits are overwritten by d(loss)/d(logits)*grad_scale.

    targets < 0 are ignored (loss 0, grad 0).  ``losses`` [M] fp32 gets the per-row loss.
    """
    lg = logits[:, :V].float()
    lse = torch.logsumexp(lg, dim=-1)
    valid = targets >= 0
    tgt = targets.clamp_min(0).long()
    picked = lg.gather(1, tgt[:, None]).squeeze(1)
    losses.copy_(torch.where(valid, lse - picked, torch.zeros_like(lse)))
    if grad_scale is not None:
        p = torch.exp(lg - lse[:, None])
        p.scatter_add_(1, tgt[:, None], -torch.ones_like(picked)[:, None])
        p = p * (valid.float() * grad_scale)[:, None]
        logits[:, :V].copy_(p.to(logits.dtype))
        if logits.shape[1] > V:
            logits[:, V:].zero_()
    return losses


def colsum(x, out):
    """out[N] (fp32) += sum over rows of x [M,N]."""
    out.add_(x.float().sum(0))
    return out


def adamw_step(master, p16, grad, m, v, *, lr, beta1, beta2, eps, weight_decay, step, decay_mask=None, grad_scale=1.0):
    """Fused multi-tensor AdamW over flat arenas (bias-corrected, ``transformers.AdamW`` semantics:
    reference hivetrain/training_manager.py:51 -> lr 5e-4, betas (0.9, 0.999), eps 1e-6, wd 0)."""
    g = grad.float() * grad_scale
    m.mul_(beta1).add_(g, alpha=1 - beta1)
    v.mul_(beta2).addcmul_(g, g, value=1 - beta2)
    bc1 = 1 - beta1 ** step
    bc2 = 1 - beta2 ** step
    step_size = lr * math.sqrt(bc2) / bc1
    master.addcdiv_(m, v.sqrt().add_(eps), value=-step_size)
    if weight_decay != 0.0:
        if decay_mask is not None:
            master.sub_(master * decay_mask, alpha=lr * weight_decay)
        else:
            master.mul_(1 - lr * weight_decay)
    if p16 is not None and p16.data_ptr() != master.data_ptr():
        p16.copy_(master.to(p16.dtype))
    return master


def delta_emit(master, base, out):
    """out = master - base (cast to out.dtype).  Reference training_manager.py:417-421 (148 separate subs)."""
    out.copy_((master.float() - base.float()).to(out.dtype))
    return out


def weighted_avg(base, deltas: Sequence[torch.Tensor], w, tensor_ids, out, nan_flags=None, delta_scales=None):
    """out = s_j * base + sum_i w[i,j] * delta_i, with s_j = sum_i w[i,j] (SURVEY 2.6-C.2).

    == sum_i w[i,j] * (base + delta_i), the reference's averaging_logic.py:434-446, in one pass.
    ``nan_flags`` [N] int32 is set to 1 for every delta containing a non-finite value (NaN screen, :121-127).
    """
    N = len(deltas)
    s = w.sum(0)  # [P]
    acc = base.float() * s[tensor_ids]
    for i in range(N):
        d = deltas[i].float()
        if delta_scales is not None:
            d = d * delta_scales[i]
        if nan_flags is not None and not torch.isfinite(d).all():
            nan_flags[i] = 1
        acc = acc + w[i][tensor_ids] * d
    out.copy_(acc.to(out.dtype))
    return out


def multi_dot(g, deltas: Sequence[torch.Tensor], base, avg, tensor_ids, P, out):
    """out[i,j] = <g_j, (base_j + delta_ij) - avg_j>  -- the meta-gradient of averaging_logic.py:513-522.

    Computed as <g_j, delta_ij> + <g_j, base_j - avg_j> (N+1 segmented dots in one pass instead of 2N rebuilds).
    """
    gf = g.float()
    common = torch.zeros(P, dtype=torch.float32, device=g.device).index_add_(0, tensor_ids, gf * (base.float() - avg.float()))
    for i, d in enumerate(deltas):
        out[i].copy_(torch.zeros(P, dtype=torch.float32, device=g.device).index_add_(0, tensor_ids, gf * d.float()) + common)
    return out


def cast_copy(src, dst):
    dst.copy_(src.to(dst.dtype))
    return dst
