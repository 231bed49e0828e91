"""Decoder-only transformer family (GPT-2, Llama and Qwen3 shapes) on flat arenas.

Two implementations of the same maths:

* :func:`oracle_loss` -- straightforward autograd PyTorch over views of a flat fp32 parameter vector.  It is the
  numerical oracle for everything else and the CPU path of the simulation (``Local*``) roles.
* :class:`TransformerEngine` -- explicit forward / backward over static buffers calling :mod:`distributedtraining_b200.ops`
  (hand-written sm_100a kernels on a B200, the PyTorch reference ops on CPU).  No autograd, no allocations in the step,
  so a whole training step is CUDA-graph capturable.

The reference contributes no model code: it calls ``transformers.GPT2LMHeadModel`` (reference
hivetrain/training_manager.py:39-46, 380-384; SURVEY.md section 3.5).  Parameter *names* follow the HF state-dict so
deltas / averaged models remain inter-operable; linear weights are stored ``[out, in]`` (K-major for the tcgen05 GEMM),
i.e. transposed w.r.t. HF GPT-2's Conv1D -- :func:`to_hf_state_dict` converts.
"""
from __future__ import annotations

import math
from dataclasses import dataclass
from typing import Dict, List, Optional, Tuple

import torch
import torch.nn.functional as F

from .. import ops
from .arena import Arena, Manifest, init_arena_


@dataclass
class ModelConfig:
    family: str = "gpt2"  # gpt2 | llama
    vocab_size: int = 50258  # GPT-2 BPE + [PAD] (reference neurons/miner.py:61-62)
    n_positions: int = 1024
    n_embd: int = 768
    n_layer: int = 12
    n_head: int = 12
    n_kv_head: Optional[int] = None
    ffn: Optional[int] = None
    eps: float = 1e-5
    rope_theta: float = 500000.0
    # RoPE frequency scaling as sorted (key, value) pairs (a tuple keeps the config hashable and comparable), e.g.
    # (("factor", 32.0), ("high_freq_factor", 4.0), ("low_freq_factor", 1.0), ("original_max_position_embeddings", 8192),
    #  ("rope_type", "llama3")); None = unscaled theta^(-2i/hd).  Only "llama3" is supported (see rope_inv_freq).
    rope_scaling: Optional[Tuple[Tuple[str, object], ...]] = None
    name: str = "gpt2"
    # embd / attn / resid dropout probability in TRAIN mode.  HF GPT-2 ships 0.1 for all three and the reference miner
    # trains with it on (reference hivetrain/training_manager.py:46 ``model.train()``); Llama configs use 0.
    dropout: float = 0.0
    # attention head dim when it is decoupled from the model width (Qwen3: n_head * head_dim != n_embd); None = n_embd / n_head
    n_head_dim: Optional[int] = None
    # Qwen3 QK-norm: an RMSNorm over every q and k head (weights [head_dim] shared across heads) between the QKV projection
    # and RoPE (llama family only)
    qk_norm: bool = False

    @property
    def head_dim(self) -> int:
        return self.n_head_dim or self.n_embd // self.n_head

    @property
    def kv_heads(self) -> int:
        return self.n_kv_head or self.n_head

    @property
    def ffn_dim(self) -> int:
        return self.ffn or 4 * self.n_embd

    @property
    def qkv_dim(self) -> int:
        return (self.n_head + 2 * self.kv_heads) * self.head_dim


PRESETS: Dict[str, ModelConfig] = {
    "gpt2": ModelConfig(name="gpt2", dropout=0.1),
    "gpt2-small": ModelConfig(name="gpt2", dropout=0.1),
    "gpt2-medium": ModelConfig(name="gpt2-medium", n_embd=1024, n_layer=24, n_head=16, dropout=0.1),
    "gpt2-tiny": ModelConfig(name="gpt2-tiny", vocab_size=512, n_positions=128, n_embd=128, n_layer=2, n_head=2),
    "llama-3.2-1b": ModelConfig(family="llama", name="llama-3.2-1b", vocab_size=128256, n_positions=131072, n_embd=2048,
                                n_layer=16, n_head=32, n_kv_head=8, ffn=8192, eps=1e-5, rope_theta=500000.0),
    # shape preset of Llama-3.2-3B (head_dim 128); its "llama3" RoPE scaling comes from config.json on import
    "llama-3.2-3b": ModelConfig(family="llama", name="llama-3.2-3b", vocab_size=128256, n_positions=131072, n_embd=3072,
                                n_layer=28, n_head=24, n_kv_head=8, ffn=8192, eps=1e-5, rope_theta=500000.0),
    "llama-tiny": ModelConfig(family="llama", name="llama-tiny", vocab_size=512, n_positions=256, n_embd=128, n_layer=2,
                              n_head=4, n_kv_head=2, ffn=256, eps=1e-5, rope_theta=10000.0),
    # Qwen3 dense models with a tied LM head: the Llama block plus QK-norm, head_dim 128 decoupled from the width, unscaled
    # RoPE (theta 1e6).  Raw vocabulary; an imported checkpoint directory gets the [PAD] row on top (get_config).
    "qwen3-0.6b": ModelConfig(family="llama", name="qwen3-0.6b", vocab_size=151936, n_positions=40960, n_embd=1024,
                              n_layer=28, n_head=16, n_kv_head=8, n_head_dim=128, ffn=3072, eps=1e-6, rope_theta=1e6,
                              qk_norm=True),
    "qwen3-1.7b": ModelConfig(family="llama", name="qwen3-1.7b", vocab_size=151936, n_positions=40960, n_embd=2048,
                              n_layer=28, n_head=16, n_kv_head=8, n_head_dim=128, ffn=6144, eps=1e-6, rope_theta=1e6,
                              qk_norm=True),
    "qwen3-4b": ModelConfig(family="llama", name="qwen3-4b", vocab_size=151936, n_positions=40960, n_embd=2560,
                            n_layer=36, n_head=32, n_kv_head=8, n_head_dim=128, ffn=9728, eps=1e-6, rope_theta=1e6,
                            qk_norm=True),
    # test shape: 4 heads x hd 64 = 256 != n_embd 128 (decoupled head dim)
    "qwen3-tiny": ModelConfig(family="llama", name="qwen3-tiny", vocab_size=512, n_positions=256, n_embd=128, n_layer=2,
                              n_head=4, n_kv_head=2, n_head_dim=64, ffn=256, eps=1e-6, rope_theta=1e6, qk_norm=True),
}


def get_config(name) -> ModelConfig:
    if isinstance(name, ModelConfig):
        return name
    import os
    if os.path.isdir(name) and os.path.exists(os.path.join(name, "config.json")):  # HF checkpoint directory (+ [PAD] row)
        import dataclasses
        import json
        with open(os.path.join(name, "config.json")) as f:
            c = config_from_hf(json.load(f))
        return dataclasses.replace(c, vocab_size=c.vocab_size + 1)
    key = name.lower().replace("openai-community/", "").replace("_", "-")
    if key not in PRESETS:
        raise KeyError(f"unknown model {name!r}; known: {sorted(PRESETS)}")
    return PRESETS[key]


# ---------------------------------------------------------------------------------------------------------------------
# manifests
# ---------------------------------------------------------------------------------------------------------------------
def build_manifest(cfg: ModelConfig) -> Manifest:
    d, Fd = cfg.n_embd, cfg.ffn_dim
    e: List[Tuple[str, Tuple[int, ...], str, bool]] = []
    if cfg.family == "gpt2":
        e.append(("transformer.wte.weight", (cfg.vocab_size, d), "normal", True))
        e.append(("transformer.wpe.weight", (cfg.n_positions, d), "normal", True))
        for l in range(cfg.n_layer):
            p = f"transformer.h.{l}."
            e += [
                (p + "ln_1.weight", (d,), "ones", False), (p + "ln_1.bias", (d,), "zeros", False),
                (p + "attn.c_attn.weight", (3 * d, d), "normal", True), (p + "attn.c_attn.bias", (3 * d,), "zeros", False),
                (p + "attn.c_proj.weight", (d, d), "normal_resid", True), (p + "attn.c_proj.bias", (d,), "zeros", False),
                (p + "ln_2.weight", (d,), "ones", False), (p + "ln_2.bias", (d,), "zeros", False),
                (p + "mlp.c_fc.weight", (Fd, d), "normal", True), (p + "mlp.c_fc.bias", (Fd,), "zeros", False),
                (p + "mlp.c_proj.weight", (d, Fd), "normal_resid", True), (p + "mlp.c_proj.bias", (d,), "zeros", False),
            ]
        e += [("transformer.ln_f.weight", (d,), "ones", False), ("transformer.ln_f.bias", (d,), "zeros", False)]
    elif cfg.family == "llama":
        hd = cfg.head_dim
        e.append(("model.embed_tokens.weight", (cfg.vocab_size, d), "normal", True))
        for l in range(cfg.n_layer):
            p = f"model.layers.{l}."
            e += [
                (p + "input_layernorm.weight", (d,), "ones", False),
                (p + "self_attn.q_proj.weight", (cfg.n_head * hd, d), "normal", True),
                (p + "self_attn.k_proj.weight", (cfg.kv_heads * hd, d), "normal", True),
                (p + "self_attn.v_proj.weight", (cfg.kv_heads * hd, d), "normal", True),
            ]
            if cfg.qk_norm:  # after v_proj: q|k|v stays one fused view, and the arena stays in program order (configure_ready)
                e += [(p + "self_attn.q_norm.weight", (hd,), "ones", False), (p + "self_attn.k_norm.weight", (hd,), "ones", False)]
            e += [
                (p + "self_attn.o_proj.weight", (d, cfg.n_head * hd), "normal_resid", True),
                (p + "post_attention_layernorm.weight", (d,), "ones", False),
                (p + "mlp.gate_proj.weight", (Fd, d), "normal", True),
                (p + "mlp.up_proj.weight", (Fd, d), "normal", True),
                (p + "mlp.down_proj.weight", (d, Fd), "normal_resid", True),
            ]
        e.append(("model.norm.weight", (d,), "ones", False))
    else:
        raise ValueError(cfg.family)
    return Manifest(e)


def fused_view(man: Manifest, flat: torch.Tensor, names: List[str]) -> torch.Tensor:
    """One [sum(rows), cols] matrix over consecutive arena tensors (q|k|v, gate|up): requires gap-free placement."""
    specs = [man[n] for n in names]
    cols = specs[0].shape[1]
    off = specs[0].offset
    rows = 0
    for s in specs:
        assert s.offset == off + rows * cols and s.shape[1] == cols, f"{s.name} is not contiguous with its group"
        rows += s.shape[0]
    return flat[off:off + rows * cols].view(rows, cols)


class LayerParams:
    """Per-layer views (compute dtype) or grad views (fp32) resolved once."""

    def __init__(self, cfg: ModelConfig, man: Manifest, flat: torch.Tensor, l: int):
        v = lambda n: man.view(flat, n)
        if cfg.family == "gpt2":
            p = f"transformer.h.{l}."
            self.ln1_w, self.ln1_b = v(p + "ln_1.weight"), v(p + "ln_1.bias")
            self.qkv_w, self.qkv_b = v(p + "attn.c_attn.weight"), v(p + "attn.c_attn.bias")
            self.o_w, self.o_b = v(p + "attn.c_proj.weight"), v(p + "attn.c_proj.bias")
            self.ln2_w, self.ln2_b = v(p + "ln_2.weight"), v(p + "ln_2.bias")
            self.fc_w, self.fc_b = v(p + "mlp.c_fc.weight"), v(p + "mlp.c_fc.bias")
            self.proj_w, self.proj_b = v(p + "mlp.c_proj.weight"), v(p + "mlp.c_proj.bias")
            self.q_norm = self.k_norm = None
        else:
            p = f"model.layers.{l}."
            self.ln1_w, self.ln1_b = v(p + "input_layernorm.weight"), None
            self.qkv_w = fused_view(man, flat, [p + "self_attn.q_proj.weight", p + "self_attn.k_proj.weight",
                                                p + "self_attn.v_proj.weight"])
            self.qkv_b = None
            self.q_norm, self.k_norm = ((v(p + "self_attn.q_norm.weight"), v(p + "self_attn.k_norm.weight")) if cfg.qk_norm
                                        else (None, None))
            self.o_w, self.o_b = v(p + "self_attn.o_proj.weight"), None
            self.ln2_w, self.ln2_b = v(p + "post_attention_layernorm.weight"), None
            self.fc_w = fused_view(man, flat, [p + "mlp.gate_proj.weight", p + "mlp.up_proj.weight"])
            self.fc_b = None
            self.proj_w, self.proj_b = v(p + "mlp.down_proj.weight"), None


class ModelParams:
    def __init__(self, cfg: ModelConfig, man: Manifest, flat: torch.Tensor):
        v = lambda n: man.view(flat, n)
        if cfg.family == "gpt2":
            self.wte, self.wpe = v("transformer.wte.weight"), v("transformer.wpe.weight")
            self.lnf_w, self.lnf_b = v("transformer.ln_f.weight"), v("transformer.ln_f.bias")
        else:
            self.wte, self.wpe = v("model.embed_tokens.weight"), None
            self.lnf_w, self.lnf_b = v("model.norm.weight"), None
        self.layers = [LayerParams(cfg, man, flat, l) for l in range(cfg.n_layer)]


# ---------------------------------------------------------------------------------------------------------------------
# autograd oracle
# ---------------------------------------------------------------------------------------------------------------------
def _norm(cfg, x, w, b):
    if cfg.family == "gpt2":
        return F.layer_norm(x, (x.shape[-1],), w, b, cfg.eps)
    rs = torch.rsqrt(x.pow(2).mean(-1, keepdim=True) + cfg.eps)
    return x * rs * w


def rope_inv_freq(cfg: ModelConfig, device=None) -> torch.Tensor:
    """fp32 [hd/2] RoPE inverse frequencies: theta^(-2i/hd), with ``cfg.rope_scaling`` applied.  "llama3" (Llama 3.1 / 3.2)
    is HF's rule (``transformers.modeling_rope_utils._compute_llama3_parameters``): wavelengths longer than
    original_max_position_embeddings / low_freq_factor are divided by ``factor``, shorter than .. / high_freq_factor kept,
    and the band in between interpolated; the attention scale is unchanged."""
    half = cfg.head_dim // 2
    inv = 1.0 / (cfg.rope_theta ** (torch.arange(0, half, device=device, dtype=torch.float32) / half))
    if cfg.rope_scaling is None:
        return inv
    sc = dict(cfg.rope_scaling)
    if sc.get("rope_type") != "llama3":
        raise ValueError(f"unsupported rope_type {sc.get('rope_type')!r}")
    factor, lo, hi = float(sc["factor"]), float(sc["low_freq_factor"]), float(sc["high_freq_factor"])
    old_ctx = float(sc["original_max_position_embeddings"])
    low_wavelen, high_wavelen = old_ctx / lo, old_ctx / hi
    wavelen = 2 * math.pi / inv
    inv_l = torch.where(wavelen > low_wavelen, inv / factor, inv)
    smooth = (old_ctx / wavelen - lo) / (hi - lo)
    smoothed = (1 - smooth) * inv_l / factor + smooth * inv_l
    medium = ~(wavelen < high_wavelen) * ~(wavelen > low_wavelen)
    return torch.where(medium, smoothed, inv_l)


def _rope(x, inv):  # x [B,T,h,hd], inv [hd/2] (rope_inv_freq)
    B, T, h, hd = x.shape
    half = hd // 2
    ang = torch.arange(T, device=x.device, dtype=torch.float32)[:, None] * inv[None, :]
    c, s = ang.cos()[None, :, None, :], ang.sin()[None, :, None, :]
    x1, x2 = x[..., :half], x[..., half:]
    return torch.cat([x1 * c - x2 * s, x2 * c + x1 * s], dim=-1)


def make_targets(input_ids: torch.Tensor, labels: Optional[torch.Tensor] = None) -> torch.Tensor:
    """HF causal-LM shift: position t predicts labels[t+1]; the last position is ignored (-1).

    The reference passes ``labels=input_ids`` with PAD *not* masked (reference neurons/miner.py:95-99,
    hivetrain/training_manager.py:383) -- we keep that: only negative labels are ignored.
    """
    lab = input_ids if labels is None else labels
    tgt = torch.full_like(lab, -1)
    tgt[..., :-1] = lab[..., 1:]
    return tgt


def drop_stream(site: str, l: int = 0) -> int:
    """Dropout site -> stream id of the counter-based mask generator (csrc/dropout.cuh)."""
    return {"embd": 0, "attn": 1 + 3 * l, "resid1": 2 + 3 * l, "resid2": 3 + 3 * l}[site]


def kv_len_of(attention_mask: Optional[torch.Tensor], T: int) -> Optional[torch.Tensor]:
    """int32 [B] count of un-padded keys per sequence from an HF ``attention_mask`` of a RIGHT-padded batch (the
    reference's tokenizer pads right: neurons/miner.py:78-92); clamped to >= 1 (an all-PAD row keeps its first key)."""
    if attention_mask is None:
        return None
    return attention_mask.reshape(-1, T).sum(dim=1).clamp_(min=1).to(torch.int32)


def oracle_logits(cfg: ModelConfig, man: Manifest, theta: torch.Tensor, input_ids: torch.Tensor,
                  drop_state=None, attention_mask: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Plain autograd forward.  ``drop_state`` (the engine's ``rng.state`` AFTER its advance, or a (seed, counter) tuple)
    turns on train-mode dropout with exactly the masks the kernels generate.  ``attention_mask`` [B,T]: padding mask as
    the reference passes it to HF GPT-2 (keys of PAD positions are invisible to every query)."""
    from ..ops import reference as ref
    P = ModelParams(cfg, man, theta)
    B, T = input_ids.shape
    H, Hkv, hd = cfg.n_head, cfg.kv_heads, cfg.head_dim
    pd = cfg.dropout if drop_state is not None else 0.0
    dm = lambda site, l=0: ref.drop_mult_2d(drop_state, drop_stream(site, l), pd, B * T, cfg.n_embd, theta.device).view(B, T, -1)
    x = P.wte[input_ids]
    if P.wpe is not None:
        x = x + P.wpe[:T][None]
    if pd > 0:
        x = x * dm("embd")
    mask = ref.attn_mask(B, T, theta.device, kv_len_of(attention_mask, T))
    inv_freq = rope_inv_freq(cfg, theta.device) if cfg.family == "llama" else None
    for l, L in enumerate(P.layers):
        h = _norm(cfg, x, L.ln1_w, L.ln1_b)
        qkv = F.linear(h, L.qkv_w, L.qkv_b)
        q, k, v = qkv.split([H * hd, Hkv * hd, Hkv * hd], dim=-1)
        q, k, v = q.view(B, T, H, hd), k.view(B, T, Hkv, hd), v.view(B, T, Hkv, hd)
        if cfg.qk_norm:  # per-head RMSNorm before RoPE (HF Qwen3Attention)
            q = q * torch.rsqrt(q.pow(2).mean(-1, keepdim=True) + cfg.eps) * L.q_norm
            k = k * torch.rsqrt(k.pow(2).mean(-1, keepdim=True) + cfg.eps) * L.k_norm
        if cfg.family == "llama":
            q, k = _rope(q, inv_freq), _rope(k, inv_freq)
        q, k, v = q.transpose(1, 2), k.transpose(1, 2), v.transpose(1, 2)
        if Hkv != H:
            k = k.repeat_interleave(H // Hkv, dim=1)
            v = v.repeat_interleave(H // Hkv, dim=1)
        s = (q @ k.transpose(-1, -2)) / math.sqrt(hd)
        s = s.masked_fill(~mask, float("-inf"))
        pr = torch.softmax(s, dim=-1)
        if pd > 0:
            pr = pr * ref.drop_mult_attn(drop_state, drop_stream("attn", l), pd, B, T, H, theta.device)
        a = (pr @ v).transpose(1, 2).reshape(B, T, H * hd)
        y = F.linear(a, L.o_w, L.o_b)
        x = x + (y * dm("resid1", l) if pd > 0 else y)
        h = _norm(cfg, x, L.ln2_w, L.ln2_b)
        u = F.linear(h, L.fc_w, L.fc_b)
        if cfg.family == "gpt2":
            act = F.gelu(u, approximate="tanh")
        else:
            g, up = u.chunk(2, dim=-1)
            act = F.silu(g) * up
        y = F.linear(act, L.proj_w, L.proj_b)
        x = x + (y * dm("resid2", l) if pd > 0 else y)
    x = _norm(cfg, x, P.lnf_w, P.lnf_b)
    return F.linear(x, P.wte)


def oracle_loss(cfg, man, theta, input_ids, labels=None, drop_state=None, attention_mask=None) -> torch.Tensor:
    logits = oracle_logits(cfg, man, theta, input_ids, drop_state, attention_mask)
    tgt = make_targets(input_ids, labels)
    return F.cross_entropy(logits.view(-1, logits.shape[-1]).float(), tgt.view(-1).long(), ignore_index=-1)


# ---------------------------------------------------------------------------------------------------------------------
# explicit engine
# ---------------------------------------------------------------------------------------------------------------------
class TransformerEngine:
    """Static-buffer forward/backward.  ``params`` is the compute-dtype arena (bf16 on GPU), ``grads`` the fp32 arena."""

    def __init__(self, cfg: ModelConfig, manifest: Manifest, params: torch.Tensor, grads: Optional[torch.Tensor],
                 batch: int, seq: int, lm_chunk: int = 8192, fp8_forward: bool = False, seed: int = 0, eval_only: bool = False,
                 fp8_backward: bool = False):
        self.cfg, self.man = cfg, manifest
        # eval_only: forward passes only -> ONE set of per-layer activation buffers shared by all layers (the validator scores
        # 51 200 tokens per miner: per-layer buffers for GPT-2-medium would be 40 GB, shared ones 1.7 GB)
        self.eval_only = bool(eval_only) and grads is None
        assert cfg.dropout == 0.0 or cfg.family == "gpt2", "dropout sites are defined for the GPT-2 family"
        self.drop_p = float(cfg.dropout)
        self.rng = ops.DropoutRng(params.device, seed=0x5EED + seed)
        self._dropping = False
        self.B, self.T, self.M = batch, seq, batch * seq
        assert seq <= cfg.n_positions
        self.dev = params.device
        self.cdtype = params.dtype
        self.P = ModelParams(cfg, manifest, params)
        self.P_flat = params
        self._delta = self._src = None
        self._src_flat = None
        self._w8_stale = True
        self.G = ModelParams(cfg, manifest, grads) if grads is not None else None
        self.grads = grads
        d, Fd, M = cfg.n_embd, cfg.ffn_dim, self.M
        mk = lambda *shape, dtype=None: torch.empty(*shape, dtype=dtype or self.cdtype, device=self.dev)
        L = cfg.n_layer
        glu = cfg.family == "llama"
        f32 = torch.float32

        def per_layer(n, *shape, dtype=None):  # n buffers, or (eval_only) one buffer aliased n times
            if self.eval_only:
                one = mk(*shape, dtype=dtype)
                return [one] * n
            return [mk(*shape, dtype=dtype) for _ in range(n)]
        if self.eval_only:
            a, b = mk(M, d), mk(M, d)
            self.xs = [a if l % 2 == 0 else b for l in range(L + 1)]  # residual stream ping-pongs between two buffers
        else:
            self.xs = [mk(M, d) for _ in range(L + 1)]  # residual stream at layer boundaries
        self.xmid = per_layer(L, M, d)
        self.h1 = per_layer(L, M, d)
        self.h2 = per_layer(L, M, d)
        self.qkv = per_layer(L, M, cfg.qkv_dim)
        self.att = per_layer(L, M, cfg.n_head * cfg.head_dim)
        self.lse = per_layer(L, batch, cfg.n_head, seq, dtype=f32)
        self.u = per_layer(L, M, 2 * Fd if glu else Fd)  # pre-activation
        self.act = per_layer(L, M, Fd)
        self.mean1 = per_layer(L, M, dtype=f32)
        self.rstd1 = per_layer(L, M, dtype=f32)
        self.mean2 = per_layer(L, M, dtype=f32)
        self.rstd2 = per_layer(L, M, dtype=f32)
        self.xf = mk(M, d)
        self.meanf, self.rstdf = mk(M, dtype=f32), mk(M, dtype=f32)
        self.lm_chunk = min(lm_chunk, M)
        self.ldl = (cfg.vocab_size + 63) // 64 * 64  # padded logits pitch (16 B aligned rows for TMA)
        self.logits = mk(self.lm_chunk, self.ldl)
        self.losses = mk(M, dtype=f32)
        self.loss = torch.zeros((), dtype=f32, device=self.dev)
        # scaled RoPE: the inverse-frequency table is built once here (the step stays capturable); unscaled configs pass no
        # table and the kernel computes theta^(-2i/hd) inline.  The fused QK-norm + RoPE kernel always reads the table.
        self.rope_inv = rope_inv_freq(cfg, self.dev) if glu and (cfg.rope_scaling is not None or cfg.qk_norm) else None
        # QK-norm saves for the backward: the raw q|k heads and their rstd (eval-only engines save nothing)
        nqk = cfg.n_head + cfg.kv_heads
        self.qk_raw = [mk(M, nqk * cfg.head_dim) for _ in range(L)] if cfg.qk_norm and not self.eval_only else None
        self.qk_rstd = [mk(M, nqk, dtype=f32) for _ in range(L)] if cfg.qk_norm and not self.eval_only else None
        # backward scratch
        if not self.eval_only:
            self.dx = mk(M, d)
            self.dx2 = mk(M, d)
            self.dxf = mk(M, d)
            if self.drop_p > 0.0 and grads is not None:
                self.dxm, self.dxm2 = mk(M, d), mk(M, d)  # dropout-masked copies of the residual-stream gradient
            self.dh = mk(M, d)
            self.dqkv = mk(M, cfg.qkv_dim)
            self.datt = mk(M, cfg.n_head * cfg.head_dim)
            self.du = mk(M, 2 * Fd if glu else Fd)
            self.dact = mk(M, Fd) if glu else None
        # ---- optional fp8 (e4m3) forward GEMMs with delayed per-tensor scaling (BASELINE.json config 4: "fp8 miners") ----
        # forward GEMM operands are quantised (weights once per step, activations by a one-pass quantise kernel that also
        # collects the amax for the NEXT step); backward GEMMs stay bf16.  All scales live in two device vectors.
        self.fp8 = bool(fp8_forward)
        # fp8 DGRAD (dX = dY W): dY quantised to e5m2 (range over precision, delayed scaling), W read from a TRANSPOSED e4m3 copy
        # (the fp8 GEMM takes K-major operands, and K = out features here); wgrad and the LM head stay bf16
        self.fp8_bwd = bool(fp8_backward) and self.fp8 and grads is not None
        if self.fp8:
            n_sc = 12 * L + 2 if self.fp8_bwd else 8 * L + 2
            self._scales = torch.full((n_sc,), 8.0 / 448.0, dtype=f32, device=self.dev)
            self._amaxes = torch.zeros(n_sc, dtype=f32, device=self.dev)

            def sc(i):
                st = ops.Fp8Scale.__new__(ops.Fp8Scale)
                st.scale, st.amax = self._scales[i:i + 1], self._amaxes[i:i + 1]
                return st
            self._sc = [sc(i) for i in range(n_sc)]
            self.w8 = torch.zeros(manifest.total, dtype=torch.uint8, device=self.dev)
            self.P8 = ModelParams(cfg, manifest, self.w8)
            self.a8 = torch.empty(M * max(2 * Fd if glu else Fd, d, cfg.qkv_dim), dtype=torch.uint8, device=self.dev)
            self._fmax = torch.full((n_sc,), 448.0, dtype=f32, device=self.dev)  # format maximum per scale slot
            if self.fp8_bwd:
                self._fmax[8 * L + 2:] = 57344.0  # e5m2 slots of the activation gradients
                self._scales[8 * L + 2:] = 1e-4    # first-step guess for gradient magnitudes (replaced by the measured amax)
                self.w8t = torch.zeros(manifest.total, dtype=torch.uint8, device=self.dev)

                def tview(w):  # [in, out] view over the arena range of weight ``w`` ([out, in], contiguous rows)
                    off = (w.data_ptr() - self.P_flat.data_ptr()) // self.P_flat.element_size()
                    return self.w8t[off:off + w.numel()].view(w.shape[1], w.shape[0])
                self.W8T = [{n: tview(getattr(self.P.layers[l], n)) for n in self._FP8_SLOTS} for l in range(L)]
        self.targets = torch.full((batch, seq), -1, dtype=torch.int32, device=self.dev)
        self.ids = torch.zeros((batch, seq), dtype=torch.int32, device=self.dev)
        # un-padded keys per sequence (HF attention_mask of a right-padded batch); = T when no mask is given.  Always passed
        # to the attention kernels so that a captured CUDA graph serves masked and unmasked batches alike.
        self.kvlen = torch.full((batch,), seq, dtype=torch.int32, device=self.dev)
        self.n_rows = batch
        self._kv_masked = False
        self.loss_denominator: Optional[int] = None  # override of the CE normaliser (data-parallel meta-learning)

    # -- helpers ---------------------------------------------------------------------------------------------------
    def _norm_fwd(self, x, w, b, out, mean, rstd):
        if self.cfg.family == "gpt2":
            ops.layernorm_fwd(x, w, b, self.cfg.eps, out, mean, rstd)
        else:
            ops.rmsnorm_fwd(x, w, self.cfg.eps, out, rstd)

    def _norm_bwd(self, dy, x, w, mean, rstd, dx_out, dw, db, dresid, dcol=None, dxm=None, drop=None):
        if self.cfg.family == "gpt2":
            ops.layernorm_bwd(dy, x, w, mean, rstd, dx_out, dw, db, dresid, dcol, dxm, drop)
        else:
            ops.rmsnorm_bwd(dy, x, w, rstd, dx_out, dw, dresid)

    def _drop(self, site: str, l: int = 0):
        return ops.Drop(self.rng, drop_stream(site, l), self.drop_p) if self._dropping else None

    def set_batch(self, input_ids, labels: Optional[torch.Tensor] = None, attention_mask: Optional[torch.Tensor] = None,
                  kv_len: Optional[torch.Tensor] = None) -> None:
        """Copy a batch into the static id/target buffers (non-blocking when the source is pinned).  A batch with fewer
        than B rows (last eval batch) is padded with ignored rows; the loss is normalised by the real row count.
        ``input_ids`` may be the reference's batch dict {"input_ids", "attention_mask", "labels"[, "kv_len"]}.
        ``attention_mask`` [B,T] (or the pre-reduced ``kv_len`` [B]) masks PAD keys exactly like HF GPT-2 does for the
        reference (training_manager.py:380-384); without it attention is causal-only."""
        if isinstance(input_ids, dict):
            d = input_ids
            input_ids = d["input_ids"]
            labels = d.get("labels", labels) if labels is None else labels
            attention_mask = d.get("attention_mask", attention_mask)
            kv_len = d.get("kv_len", kv_len)
        ids2 = input_ids.view(-1, self.T)
        n = ids2.shape[0]
        assert n <= self.B, f"batch of {n} rows exceeds the engine's static batch {self.B}"
        self.n_rows = n
        src = ids2 if labels is None else labels.view(-1, self.T)
        if n < self.B:
            self.ids[n:].zero_()
            self.targets[n:].fill_(-1)
        self.ids[:n].copy_(ids2, non_blocking=True)
        self.targets[:n, :-1].copy_(src[:, 1:], non_blocking=True)
        if kv_len is None and attention_mask is not None:
            kv_len = kv_len_of(attention_mask, self.T)
        if kv_len is not None:
            self.kvlen[:n].copy_(kv_len.view(-1)[:n], non_blocking=True)
            if n < self.B:
                self.kvlen[n:].fill_(self.T)
        elif self._kv_masked:
            self.kvlen.fill_(self.T)
        self._kv_masked = kv_len is not None

    # -- forward ---------------------------------------------------------------------------------------------------
    def set_delta(self, delta_flat: Optional[torch.Tensor]) -> None:
        """Fused delta evaluation (validator): every weight GEMM computes ``x (W + dW)^T`` as two accumulating tensor-core
        passes with ``dW`` read straight from ``delta_flat`` (bf16, may live in a miner's PEER window) and the embedding
        adds the delta rows on the fly -- ``theta_base + delta_i`` is never materialised for the matrices.  The small
        tensors (norm weights, biases) must already hold base+delta in the compute arena (see ``small_chunk_ids``)."""
        self._delta = None if delta_flat is None else ModelParams(self.cfg, self.man, delta_flat)

    def set_source(self, src_flat: Optional[torch.Tensor]) -> None:
        """Fused broadcast -> first forward: weights are read from ``src_flat`` (the averager's bf16 window over NVLink)
        and every B tile is persisted into this rank's compute arena by the GEMM that consumes it."""
        self._src = None if src_flat is None else ModelParams(self.cfg, self.man, src_flat)
        self._src_flat = src_flat

    # -- fused broadcast -> first forward GEMM (path (b)) -----------------------------------------------------------------
    _FWD_GEMMS = ("qkv_w", "o_w", "fc_w", "proj_w")

    def configure_ready(self, flags_address: int, target: torch.Tensor, chunks_per_rank: int, world: int) -> None:
        """The weights of a NEW averaged base are landed in this arena by the shard owners' averaging kernels (rank k owns the
        chunks [k*per, (k+1)*per) of the chunk table).  In ``ready`` mode every forward GEMM acquires, inside the kernel, the
        base flags of the owners of everything that is consumed up to the next GEMM (its own weight and bias, the following
        norm weights, ...): the arena is laid out in program order, so the owners a GEMM has to wait for are 0..need.  The
        tensors consumed before the first GEMM (embedding tables, first norm) are covered by one tiny wait kernel."""
        cs, _, _ = self.man.seg_table("cpu")
        esz = self.P_flat.element_size()

        def owner_before(view) -> int:  # owner of the arena element right before ``view`` starts
            e = (view.data_ptr() - self.P_flat.data_ptr()) // esz - 1
            if e < 0:
                return 0
            c = int(torch.searchsorted(cs, torch.tensor([e], dtype=cs.dtype), right=True)) - 1
            return min(c // chunks_per_rank, world - 1)
        order = [(l, n) for l in range(self.cfg.n_layer) for n in self._FWD_GEMMS]
        views = [getattr(self.P.layers[l], n) for l, n in order]
        need = {}
        for i, key in enumerate(order):
            need[key] = owner_before(views[i + 1]) if i + 1 < len(order) else world - 1
        self._ready_need = need
        self._ready_pre = owner_before(views[0])
        self._ready_args = (flags_address, target)
        self._ready_on = False

    def _ready_for(self, l, name):
        if not getattr(self, "_ready_on", False) or l is None:
            return None
        return (self._ready_args[0], self._ready_args[1], self._ready_need[(l, name)])

    def small_chunk_ids(self) -> torch.Tensor:
        """Chunk-table indices of the non-matrix tensors (norm weights, biases, positional table)."""
        if getattr(self, "_small_ids", None) is None:
            _, _, ct = self.man.seg_table(self.dev)
            small = torch.tensor([len(s.shape) < 2 or s.name.endswith("wpe.weight") for s in self.man.specs], device=self.dev)
            self._small_ids = torch.nonzero(small[ct.long()]).flatten().to(torch.int32)
        return self._small_ids

    _FP8_SLOTS = {"qkv_w": 0, "o_w": 1, "fc_w": 2, "proj_w": 3}

    def _fgemm(self, l: Optional[int], name: str, a, out, **kw):
        """Forward GEMM ``out = epi(a @ W^T)``: bf16 tcgen05 path, or e4m3 operands when ``fp8_forward`` is on."""
        if not self.fp8 or self._delta is not None or self._src is not None:
            g = self._w(l, name)
            return ops.gemm(a, g.pop("b"), out, **g, ready=self._ready_for(l, name), **kw)
        L = self.cfg.n_layer
        slot = 8 * l + 2 * self._FP8_SLOTS[name] if l is not None else 8 * L
        sa, sw = self._sc[slot], self._sc[slot + 1]
        w = getattr(self.P.layers[l], name) if l is not None else self.P.wte
        w8 = getattr(self.P8.layers[l], name) if l is not None else self.P8.wte
        if self._w8_stale:
            ops.quantize_fp8(w, w8, sw)
            if self.fp8_bwd and l is not None:
                ops.quantize_fp8_t(w, self.W8T[l][name], sw)  # same scale, transposed layout: B operand of the dgrad
        a8 = self.a8[:a.numel()].view(a.shape)
        ops.quantize_fp8(a, a8, sa)
        return ops.gemm_fp8(a8, w8, out, sa, sw, **kw)

    _DY_SLOTS = {"proj_w": 0, "fc_w": 1, "o_w": 2, "qkv_w": 3}

    def _dgemm(self, l: int, name: str, dy, out, **kw):
        """Backward data GEMM ``out = epi(dy @ W)``: bf16 (W read MN-major), or fp8 -- dy -> e5m2, W^T from the transposed e4m3
        copy written by this step's forward."""
        w = getattr(self.P.layers[l], name)
        if not self.fp8_bwd:
            return ops.gemm(dy, w, out, b_mn=True, **kw)
        L = self.cfg.n_layer
        sdy = self._sc[8 * L + 2 + 4 * l + self._DY_SLOTS[name]]
        sw = self._sc[8 * l + 2 * self._FP8_SLOTS[name] + 1]
        dy8 = self.a8[:dy.numel()].view(dy.shape)
        ops.quantize_fp8(dy, dy8, sdy, e5m2=True)
        return ops.gemm_fp8(dy8, self.W8T[l][name], out, sdy, sw, a_e5m2=True, **kw)

    def roll_fp8_scales(self) -> None:
        """Delayed scaling: scale <- amax / 448 for the next step (3 vectorised device ops for all tensors)."""
        if self.fp8:
            torch.clamp(self._amaxes, min=1e-8, out=self._scales)
            self._scales.div_(self._fmax)
            self._amaxes.zero_()

    def _w(self, l: Optional[int], name: str) -> dict:
        """kwargs (b, b2, b_persist) of the weight operand ``name`` of layer ``l`` (None = model level)."""
        pick = (lambda P: getattr(P.layers[l], name)) if l is not None else (lambda P: getattr(P, name))
        delta, src = getattr(self, "_delta", None), getattr(self, "_src", None)
        if src is not None:
            return {"b": pick(src), "b_persist": pick(self.P)}
        if delta is not None:
            return {"b": pick(self.P), "b2": pick(delta)}
        return {"b": pick(self.P)}

    def forward(self, train: bool = True) -> None:
        cfg = self.cfg
        self._w8_stale = True  # weights may have changed since the last forward: re-quantise them on first use
        delta, src = getattr(self, "_delta", None), getattr(self, "_src", None)
        P = src if src is not None else self.P  # small tensors (norms, biases, embeddings) are read where the weights are
        B, T, H, Hkv, hd = self.B, self.T, cfg.n_head, cfg.kv_heads, cfg.head_dim
        self._dropping = bool(train and self.drop_p > 0.0)
        if self._dropping:
            self.rng.advance()  # fresh masks every training forward; backward regenerates them from the same counter
        if getattr(self, "_ready_on", False):  # embedding tables + first norm: owners 0.._ready_pre must have landed
            ops.wait_flags_dev(self._ready_args[0], self._ready_pre + 1, self._ready_args[1])
        # the position table belongs to the small set (already base+delta in the arena): only the token rows are added here
        ops.embed_fwd(self.ids, P.wte, P.wpe, self.xs[0], *((delta.wte, None) if delta is not None else ()),
                      drop=self._drop("embd"))
        for l, Lp in enumerate(P.layers):
            x = self.xs[l]
            self._norm_fwd(x, Lp.ln1_w, Lp.ln1_b, self.h1[l], self.mean1[l], self.rstd1[l])
            self._fgemm(l, "qkv_w", self.h1[l], self.qkv[l], epi="bias" if Lp.qkv_b is not None else "none", bias=Lp.qkv_b)
            if cfg.qk_norm:
                ops.qk_norm_rope_fwd(self.qkv[l], B, T, H, Hkv, hd, Lp.q_norm, Lp.k_norm, cfg.eps, self.rope_inv,
                                     *((self.qk_raw[l], self.qk_rstd[l]) if self.qk_raw is not None else ()))
            elif cfg.family == "llama":
                ops.rope_(self.qkv[l], B, T, H, Hkv, hd, cfg.rope_theta, inv_freq=self.rope_inv)
            ops.attention_fwd(self.qkv[l], self.att[l], self.lse[l], B, T, H, hd, Hkv, drop=self._drop("attn", l),
                              kv_len=self.kvlen)
            self._fgemm(l, "o_w", self.att[l], self.xmid[l], epi="bias_resid" if Lp.o_b is not None else "resid", bias=Lp.o_b,
                        aux=x, drop=self._drop("resid1", l))
            self._norm_fwd(self.xmid[l], Lp.ln2_w, Lp.ln2_b, self.h2[l], self.mean2[l], self.rstd2[l])
            if cfg.family == "gpt2":
                self._fgemm(l, "fc_w", self.h2[l], self.act[l], epi="bias_gelu", bias=Lp.fc_b, out2=self.u[l])
            else:
                self._fgemm(l, "fc_w", self.h2[l], self.u[l])
                ops.swiglu_fwd(self.u[l], self.act[l])
            self._fgemm(l, "proj_w", self.act[l], self.xs[l + 1], epi="bias_resid" if Lp.proj_b is not None else "resid",
                        bias=Lp.proj_b, aux=self.xmid[l], drop=self._drop("resid2", l))
        self._norm_fwd(self.xs[-1], P.lnf_w, P.lnf_b, self.xf, self.meanf, self.rstdf)

    def _lm_head(self, backward: bool) -> None:
        cfg, P = self.cfg, self.P
        V = cfg.vocab_size
        n_valid = self.loss_denominator if self.loss_denominator is not None else self.n_rows * (self.T - 1)
        scale = 1.0 / max(n_valid, 1)
        tgt = self.targets.view(-1)
        first = True
        for c0 in range(0, self.M, self.lm_chunk):
            c1 = min(self.M, c0 + self.lm_chunk)
            lg = self.logits[:c1 - c0]  # [rows, ldl] padded pitch; lgv is the logical [rows, V] view (TMA clips/zero-fills)
            lgv = lg[:, :V]
            g = self._w(None, "wte")
            if not first:
                g.pop("b_persist", None)  # the first chunk's GEMM already persisted the table
                if getattr(self, "_src", None) is not None:
                    g["b"] = P.wte
            ops.gemm(self.xf[c0:c1], g.pop("b"), lgv, **g)
            first = False
            ops.ce_fwd_bwd(lg, tgt[c0:c1], V, self.losses[c0:c1], scale if backward else None)
            if backward:
                ops.gemm(lgv, P.wte, self.dxf[c0:c1], b_mn=True)  # dxf = dlogits @ wte
                ops.gemm(lgv, self.xf[c0:c1], self.G.wte, a_mn=True, b_mn=True, accumulate=True)  # dwte += dlogits^T xf
        ops.loss_mean(self.losses, scale, self.loss)

    def persist_small_from_source(self) -> None:
        """Copy the non-matrix tensors (norms, biases, position table: < 1 % of the bytes) from the peer source."""
        src = getattr(self, "_src", None)
        if src is None:
            return
        for s in self.man.specs:
            if len(s.shape) < 2 or s.name.endswith("wpe.weight"):
                self.man.view(self.P_flat, s.name).copy_(self.man.view(self._src_flat, s.name), non_blocking=True)

    def forward_loss(self) -> torch.Tensor:
        """Eval forward: mean next-token CE over the batch in the static buffers (device scalar)."""
        self.forward(train=False)
        self._lm_head(backward=False)
        return self.loss

    # -- backward --------------------------------------------------------------------------------------------------
    def forward_backward(self, zero_grad: bool = True, dropout: bool = True) -> torch.Tensor:
        """Loss + gradients of the batch in the static buffers.  ``dropout=False`` gives the deterministic (eval-mode)
        gradient -- used by the averager's meta-learning unless ``--meta_dropout`` asks for the reference's behaviour
        (its averager keeps the model in train mode, neurons/averager.py:69)."""
        cfg, P, G = self.cfg, self.P, self.G
        B, T, H, Hkv, hd = self.B, self.T, cfg.n_head, cfg.kv_heads, cfg.head_dim
        if zero_grad:
            ops.zero_(self.grads)
        self.forward(train=dropout)
        self._lm_head(backward=True)
        # Residual-stream gradients ping-pong between dx / dx2.  Each norm backward also produces, on the same pass, what
        # the NEXT GEMM pair in the backward order needs: its dY (a dropout-masked copy when the site is active, the
        # residual gradient itself otherwise) and that GEMM's bias gradient (column sums of the dY).
        L = cfg.n_layer
        dx, dx2 = self.dx, self.dx2
        dm, dm2 = (self.dxm, self.dxm2) if self._dropping else (None, None)
        self._norm_bwd(self.dxf, self.xs[-1], P.lnf_w, self.meanf, self.rstdf, dx, G.lnf_w, G.lnf_b, None,
                       G.layers[L - 1].proj_b, dm, self._drop("resid2", L - 1))
        for l in range(L - 1, -1, -1):
            Lp, Lg = P.layers[l], G.layers[l]
            dy = dm if dm is not None else dx
            # ---- MLP block ----
            if cfg.family == "gpt2":
                self._dgemm(l, "proj_w", dy, self.du, epi="dgelu", aux=self.u[l])
            else:
                self._dgemm(l, "proj_w", dy, self.dact)
                ops.swiglu_bwd(self.dact, self.u[l], self.du)
            ops.gemm(dy, self.act[l], Lg.proj_w, a_mn=True, b_mn=True, accumulate=True)
            self._dgemm(l, "fc_w", self.du, self.dh)
            ops.gemm(self.du, self.h2[l], Lg.fc_w, a_mn=True, b_mn=True, accumulate=True)
            if Lg.fc_b is not None:
                # (folding this column sum into the dgelu GEMM's epilogue -- ops.gemm(colsum_out=...) -- was measured slower:
                # +36 us per GEMM for the smem column pass vs the 21 us of this separate launch)
                ops.colsum(self.du, Lg.fc_b)
            self._norm_bwd(self.dh, self.xmid[l], Lp.ln2_w, self.mean2[l], self.rstd2[l], dx2, Lg.ln2_w, Lg.ln2_b, dx, Lg.o_b,
                           dm2, self._drop("resid1", l))
            dx, dx2 = dx2, dx
            dm, dm2 = dm2, dm
            dy = dm if dm is not None else dx
            # ---- attention block ----
            self._dgemm(l, "o_w", dy, self.datt)
            ops.gemm(dy, self.att[l], Lg.o_w, a_mn=True, b_mn=True, accumulate=True)
            # d(qkv bias) = colsum(dqkv) rides on the attention backward (GPT-2 has no RoPE between the two)
            ops.attention_bwd(self.datt, self.qkv[l], self.att[l], self.lse[l], self.dqkv, B, T, H, hd, Hkv,
                              drop=self._drop("attn", l), dbias=Lg.qkv_b, kv_len=self.kvlen)
            if cfg.qk_norm:
                ops.qk_norm_rope_bwd(self.dqkv, B, T, H, Hkv, hd, Lp.q_norm, Lp.k_norm, self.rope_inv, self.qk_raw[l],
                                     self.qk_rstd[l], Lg.q_norm, Lg.k_norm)
            elif cfg.family == "llama":
                ops.rope_(self.dqkv, B, T, H, Hkv, hd, cfg.rope_theta, inverse=True, inv_freq=self.rope_inv)
            self._dgemm(l, "qkv_w", self.dqkv, self.dh)
            ops.gemm(self.dqkv, self.h1[l], Lg.qkv_w, a_mn=True, b_mn=True, accumulate=True)
            nxt = l - 1
            self._norm_bwd(self.dh, self.xs[l], Lp.ln1_w, self.mean1[l], self.rstd1[l], dx2, Lg.ln1_w, Lg.ln1_b, dx,
                           G.layers[nxt].proj_b if nxt >= 0 else None, dm2 if nxt >= 0 else None,
                           self._drop("resid2", nxt) if nxt >= 0 else None)
            dx, dx2 = dx2, dx
            dm, dm2 = dm2, dm
        ops.embed_bwd(dx, self.ids, G.wte, G.wpe, drop=self._drop("embd"))
        return self.loss


_CONV1D = ("c_attn.weight", "c_proj.weight", "c_fc.weight")  # HF GPT-2 stores these [in, out]; the engine [out, in]


def to_hf_state_dict(cfg: ModelConfig, arena) -> Dict[str, torch.Tensor]:
    """HF-compatible state dict (GPT-2 Conv1D weights transposed back to [in, out]; tied lm_head added -> 149 keys):
    loads straight into ``transformers.GPT2LMHeadModel`` / ``LlamaForCausalLM`` / ``Qwen3ForCausalLM`` -- the reference's checkpoint format
    (``model.state_dict()``, hivetrain/averaging_logic.py:481-488).  ``arena``: an :class:`Arena` or a flat tensor."""
    if isinstance(arena, torch.Tensor):
        arena = Arena(build_manifest(cfg), flat=arena)
    sd = arena.state_dict(clone=True)
    if cfg.family == "gpt2":
        for k in list(sd):
            if k.endswith(_CONV1D):
                sd[k] = sd[k].t().contiguous()
        sd["lm_head.weight"] = sd["transformer.wte.weight"]
    else:
        sd["lm_head.weight"] = sd["model.embed_tokens.weight"]
    return sd


def is_hf_layout(cfg: ModelConfig, sd: Dict[str, torch.Tensor]) -> bool:
    """HF GPT-2 layout is recognisable by the (non-square) c_attn weight being [d, 3d]; Llama layouts coincide."""
    if cfg.family != "gpt2":
        return True
    w = sd.get("transformer.h.0.attn.c_attn.weight")
    return w is not None and tuple(w.shape) == (cfg.n_embd, 3 * cfg.n_embd)


def from_hf_state_dict(cfg: ModelConfig, sd: Dict[str, torch.Tensor], man: Optional[Manifest] = None,
                       out: Optional[torch.Tensor] = None, resize_vocab: bool = True) -> torch.Tensor:
    """HF state dict (``GPT2LMHeadModel`` / ``LlamaForCausalLM`` / ``Qwen3ForCausalLM`` naming, or this engine's own layout)
    -> flat fp32 arena.

    * GPT-2 Conv1D weights are transposed to the engine's ``[out, in]`` (the square ``attn.c_proj`` cannot be told apart
      by shape -- the layout is detected on ``c_attn`` and applied to all of them);
    * ``lm_head.weight`` (tied) and the non-parameter buffers (``attn.bias`` / ``masked_bias``) are dropped;
    * ``resize_vocab``: a checkpoint with FEWER embedding rows than ``cfg.vocab_size`` is grown the way the reference does
      after adding ``[PAD]`` (``resize_token_embeddings``, hivetrain/training_manager.py:39-46): the new rows are set to
      the mean of the existing embeddings (HF's ``mean_resizing`` without the sampled covariance term, so that every rank
      derives the SAME base without communication);
    * every other shape mismatch raises (the reference's shape screen, averaging_logic.py:406-410).
    """
    man = man or build_manifest(cfg)
    out = out if out is not None else torch.zeros(man.total, dtype=torch.float32)
    hf = is_hf_layout(cfg, sd)
    emb = "transformer.wte.weight" if cfg.family == "gpt2" else "model.embed_tokens.weight"
    for spec in man.specs:
        if spec.name not in sd:
            raise KeyError(f"checkpoint lacks {spec.name}")
        t = sd[spec.name].detach().to(torch.float32)
        if hf and cfg.family == "gpt2" and spec.name.endswith(_CONV1D):
            t = t.t()
        if spec.name == emb and resize_vocab and t.shape[0] < spec.shape[0] and t.shape[1:] == spec.shape[1:]:
            grown = t.mean(dim=0, keepdim=True).expand(spec.shape[0], -1).clone()
            grown[:t.shape[0]] = t
            t = grown
        if tuple(t.shape) != spec.shape:
            raise ValueError(f"{spec.name}: checkpoint shape {tuple(sd[spec.name].shape)} does not fit {spec.shape}")
        out[spec.offset:spec.offset + spec.numel].copy_(t.reshape(-1))
    return out


def pack_any(man: Manifest, blob, cfg: Optional[ModelConfig] = None) -> torch.Tensor:
    """Flat fp32 arena from whatever a peer handed over: a flat tensor, an engine-layout dict, or (with ``cfg``) an HF /
    reference-format state dict (``averaged_model.pt``, ``weight_diff.pt``, ``gradients.pt``).  Wrong shapes raise."""
    if isinstance(blob, torch.Tensor):
        if blob.numel() != man.total:
            raise ValueError(f"flat tensor of {blob.numel()} elements does not fit the manifest ({man.total})")
        return blob
    if cfg is not None:
        return from_hf_state_dict(cfg, blob, man, resize_vocab=False)
    return man.pack(blob, torch.zeros(man.total, dtype=torch.float32))


def _rope_from_hf(d: dict) -> Tuple[float, Optional[Tuple[Tuple[str, object], ...]]]:
    """(theta, scaling) of an HF Llama config in either layout: top-level ``rope_theta`` / ``rope_scaling`` (transformers 4)
    or ``rope_parameters`` (transformers >= 5).  No type or "default" = unscaled; "llama3" is kept; anything else raises."""
    rp = d.get("rope_parameters") or {}
    theta = float(rp.get("rope_theta", d.get("rope_theta", 10000.0)))
    sc = d.get("rope_scaling") or (rp if "rope_type" in rp or "type" in rp else None)
    if not sc:
        return theta, None
    rt = sc.get("rope_type", sc.get("type", "default"))
    if rt == "default":
        return theta, None
    if rt != "llama3":
        raise ValueError(f"unsupported RoPE scaling type {rt!r} (supported: default, llama3)")
    keep = ("factor", "low_freq_factor", "high_freq_factor", "original_max_position_embeddings")
    missing = [k for k in keep if k not in sc]
    if missing:
        raise ValueError(f"llama3 RoPE scaling lacks {missing}")
    vals = {k: float(sc[k]) for k in keep}
    vals["original_max_position_embeddings"] = int(sc["original_max_position_embeddings"])
    vals["rope_type"] = "llama3"
    return theta, tuple(sorted(vals.items()))


def config_from_hf(d: dict) -> ModelConfig:
    """``config.json`` of an HF GPT-2 / Llama / Qwen3 checkpoint -> ModelConfig.

    Llama: RoPE theta and "llama3" scaling are read from either config layout (:func:`_rope_from_hf`); ``head_dim``, when
    present, must equal hidden_size / num_attention_heads; the LM head must be tied to the embedding
    (``tie_word_embeddings``, False when absent as in ``transformers.LlamaConfig``) -- an untied head has no place in the
    arena, and loading it as tied would silently be a different model.

    Qwen3 (dense): the Llama block with QK-norm and a ``head_dim`` that may differ from hidden_size / num_attention_heads.
    Refused with a ValueError naming the field: an untied LM head (``Qwen3Config`` defaults ``tie_word_embeddings`` to
    False), ``attention_bias``, sliding-window attention (``use_sliding_window`` or a ``layer_types`` entry other than
    full_attention), a ``hidden_act`` other than silu and RoPE scaling other than llama3 (YaRN)."""
    mt = d.get("model_type", "gpt2")
    if mt == "gpt2":
        return ModelConfig(family="gpt2", name=d.get("_name_or_path") or "gpt2-hf", vocab_size=int(d["vocab_size"]),
                           n_positions=int(d.get("n_positions", 1024)), n_embd=int(d["n_embd"]), n_layer=int(d["n_layer"]),
                           n_head=int(d["n_head"]), ffn=d.get("n_inner") or None, eps=float(d.get("layer_norm_epsilon", 1e-5)),
                           dropout=float(d.get("resid_pdrop", 0.1)))
    if mt == "llama":
        d_model, n_head = int(d["hidden_size"]), int(d["num_attention_heads"])
        if d.get("head_dim") is not None and int(d["head_dim"]) * n_head != d_model:
            raise ValueError(f"head_dim {d['head_dim']} != hidden_size / num_attention_heads = {d_model} / {n_head}: "
                             "a decoupled head dim is not supported")
        if not d.get("tie_word_embeddings", False):
            raise ValueError("tie_word_embeddings is false: an untied LM head is not supported")
        theta, scaling = _rope_from_hf(d)
        return ModelConfig(family="llama", name=d.get("_name_or_path") or "llama-hf", vocab_size=int(d["vocab_size"]),
                           n_positions=int(d.get("max_position_embeddings", 8192)), n_embd=d_model,
                           n_layer=int(d["num_hidden_layers"]), n_head=n_head,
                           n_kv_head=int(d.get("num_key_value_heads") or n_head),
                           ffn=int(d["intermediate_size"]), eps=float(d.get("rms_norm_eps", 1e-5)),
                           rope_theta=theta, rope_scaling=scaling)
    if mt == "qwen3":
        d_model, n_head = int(d["hidden_size"]), int(d["num_attention_heads"])
        if not d.get("tie_word_embeddings", False):
            raise ValueError("tie_word_embeddings is false: an untied LM head is not supported")
        if d.get("attention_bias", False):
            raise ValueError("attention_bias is true: q/k/v/o projection biases are not supported")
        if d.get("use_sliding_window", False):
            raise ValueError("use_sliding_window is true: sliding-window attention is not supported")
        bad = [t for t in (d.get("layer_types") or []) if t != "full_attention"]
        if bad:
            raise ValueError(f"layer_types holds {sorted(set(bad))}: only full_attention layers are supported")
        if d.get("hidden_act", "silu") != "silu":
            raise ValueError(f"hidden_act {d['hidden_act']!r} is not supported (silu only)")
        theta, scaling = _rope_from_hf(d)
        return ModelConfig(family="llama", name=d.get("_name_or_path") or "qwen3-hf", vocab_size=int(d["vocab_size"]),
                           n_positions=int(d.get("max_position_embeddings", 32768)), n_embd=d_model,
                           n_layer=int(d["num_hidden_layers"]), n_head=n_head,
                           n_kv_head=int(d.get("num_key_value_heads") or n_head),
                           n_head_dim=int(d.get("head_dim") or d_model // n_head), ffn=int(d["intermediate_size"]),
                           eps=float(d.get("rms_norm_eps", 1e-6)), rope_theta=theta, rope_scaling=scaling, qk_norm=True)
    raise ValueError(f"unsupported HF model_type {mt!r}")


def load_hf_checkpoint(path: str, add_pad_token: bool = True) -> Tuple[ModelConfig, Manifest, torch.Tensor]:
    """Read an HF checkpoint DIRECTORY (``config.json`` + ``model.safetensors`` | ``pytorch_model.bin``) without
    instantiating a ``transformers`` model.  ``add_pad_token`` grows the vocabulary by one row, as every reference role
    does (``tokenizer.add_special_tokens({'pad_token': '[PAD]'})`` + ``resize_token_embeddings``, neurons/miner.py:60-62)."""
    import json
    import os
    with open(os.path.join(path, "config.json")) as f:
        cfg = config_from_hf(json.load(f))
    st = os.path.join(path, "model.safetensors")
    if os.path.exists(st):
        from safetensors.torch import load_file
        sd = load_file(st)
    else:
        sd = torch.load(os.path.join(path, "pytorch_model.bin"), map_location="cpu", weights_only=True)
    if cfg.family == "gpt2" and not any(k.startswith("transformer.") for k in sd):
        sd = {"transformer." + k: v for k, v in sd.items()}  # bare GPT2Model checkpoints
    if add_pad_token:
        import dataclasses
        cfg = dataclasses.replace(cfg, vocab_size=cfg.vocab_size + 1)
    man = build_manifest(cfg)
    return cfg, man, from_hf_state_dict(cfg, sd, man)


def new_model(name_or_cfg, device="cpu", dtype=torch.float32, seed: int = 0) -> Tuple[ModelConfig, Manifest, Arena]:
    cfg = get_config(name_or_cfg) if isinstance(name_or_cfg, str) else name_or_cfg
    man = build_manifest(cfg)
    arena = Arena(man, dtype=torch.float32, device="cpu")
    init_arena_(arena, n_layer=cfg.n_layer, seed=seed)
    if str(device) != "cpu" or dtype != torch.float32:
        arena = Arena(man, flat=arena.flat.to(device=device, dtype=dtype))
    return cfg, man, arena
