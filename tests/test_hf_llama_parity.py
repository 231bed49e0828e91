"""Llama import parity against ``transformers.LlamaForCausalLM``: head_dim 128, GQA 2:1, tied embedding and Llama-3 ("llama3")
RoPE frequency scaling, read from both config layouts (transformers 4: top-level ``rope_theta`` / ``rope_scaling``;
transformers >= 5: ``rope_parameters``); the config screens; the RoPE kernel's frequency table."""
import dataclasses
import os

import pytest
import torch

transformers = pytest.importorskip("transformers")

from distributedtraining_b200 import ops
from distributedtraining_b200.models.trainer import Trainer
from distributedtraining_b200.models.transformer import (ModelConfig, build_manifest, config_from_hf, from_hf_state_dict,
                                                         get_config, oracle_loss, rope_inv_freq)
from distributedtraining_b200.ops import reference as ref

VOCAB = 300
SCALING = {"rope_type": "llama3", "factor": 8.0, "low_freq_factor": 1.0, "high_freq_factor": 4.0,
           "original_max_position_embeddings": 64}


def _hf_llama(vocab=VOCAB, d=256, L=2, H=2, Hkv=1, ffn=384, npos=256, theta=500000.0, seed=0):
    from transformers import LlamaConfig, LlamaForCausalLM
    torch.manual_seed(seed)
    cfg = LlamaConfig(vocab_size=vocab, hidden_size=d, intermediate_size=ffn, num_hidden_layers=L, num_attention_heads=H,
                      num_key_value_heads=Hkv, max_position_embeddings=npos, rms_norm_eps=1e-5, tie_word_embeddings=True,
                      rope_parameters=dict(SCALING, rope_theta=theta), attn_implementation="eager")
    m = LlamaForCausalLM(cfg).eval()
    with torch.no_grad():  # HF ones-inits the RMSNorm weights: randomise so that layout mistakes cannot hide
        for n, p in m.named_parameters():
            if p.dim() == 1:
                p.add_(0.05 * torch.randn_like(p))
    return m


def _legacy(d: dict) -> dict:
    """The same config as transformers 4 writes it: rope_theta / rope_scaling at the top level."""
    d = dict(d)
    rp = dict(d.pop("rope_parameters"))
    d["rope_theta"] = rp.pop("rope_theta")
    d["rope_scaling"] = rp
    return d


def _batch(B=4, T=128, vocab=VOCAB, pad=VOCAB - 1, seed=1):
    g = torch.Generator().manual_seed(seed)
    ids = torch.randint(0, pad, (B, T), generator=g)
    lens = torch.tensor([T, T - 37, 9, 1])[:B]
    am = (torch.arange(T)[None] < lens[:, None]).long()
    return torch.where(am.bool(), ids, torch.full_like(ids, pad)), am


def test_config_layouts_and_screens():
    m = _hf_llama()
    d5 = m.config.to_dict()
    c5, c4 = config_from_hf(d5), config_from_hf(_legacy(d5))
    assert c5 == c4
    assert c5.head_dim == 128 and c5.kv_heads == 1 and c5.rope_theta == 500000.0
    assert dict(c5.rope_scaling)["rope_type"] == "llama3"
    assert dict(c5.rope_scaling)["original_max_position_embeddings"] == 64
    # "default" (or no type) = unscaled
    plain = _legacy(d5)
    plain["rope_scaling"] = {"rope_type": "default"}
    assert config_from_hf(plain).rope_scaling is None
    plain["rope_scaling"] = None
    assert config_from_hf(plain).rope_scaling is None
    d5p = dict(d5, rope_parameters={"rope_type": "default", "rope_theta": 1234.0})
    assert config_from_hf(d5p).rope_scaling is None and config_from_hf(d5p).rope_theta == 1234.0
    # unsupported scaling types name the type
    for rt in ("linear", "dynamic", "yarn"):
        with pytest.raises(ValueError, match=rt):
            config_from_hf(dict(d5, rope_parameters=dict(d5["rope_parameters"], rope_type=rt)))
        with pytest.raises(ValueError, match=rt):
            config_from_hf(dict(_legacy(d5), rope_scaling=dict(SCALING, rope_type=rt)))
    # a decoupled head_dim and an untied LM head are refused
    with pytest.raises(ValueError, match="head_dim"):
        config_from_hf(dict(d5, head_dim=64))
    assert config_from_hf(dict(d5, head_dim=128)) == c5
    with pytest.raises(ValueError, match="tie_word_embeddings"):
        config_from_hf(dict(d5, tie_word_embeddings=False))
    # the 3B shape preset: head_dim 128, 24 / 8 heads, no scaling (it comes from config.json on import)
    p3 = get_config("llama-3.2-3b")
    assert (p3.head_dim, p3.n_head, p3.kv_heads, p3.n_layer, p3.ffn_dim, p3.vocab_size) == (128, 24, 8, 28, 8192, 128256)
    assert p3.rope_scaling is None and p3.rope_theta == 500000.0
    assert get_config("llama-3.2-1b").head_dim == 64


def test_rope_inv_freq_matches_hf():
    from transformers.modeling_rope_utils import ROPE_INIT_FUNCTIONS
    m = _hf_llama()
    want, attn_scale = ROPE_INIT_FUNCTIONS["llama3"](m.config, torch.device("cpu"))
    cfg = config_from_hf(m.config.to_dict())
    got = rope_inv_freq(cfg)
    assert attn_scale == 1.0
    assert torch.equal(got, want.float())
    unscaled = rope_inv_freq(dataclasses.replace(cfg, rope_scaling=None))
    assert not torch.equal(got, unscaled)  # the scaling really changes frequencies at this context length


@pytest.mark.parametrize("layout", ["v5", "v4"])
def test_loss_and_grads_match_hf_llama(layout):
    m = _hf_llama()
    d = m.config.to_dict()
    mc = config_from_hf(d if layout == "v5" else _legacy(d))
    man = build_manifest(mc)
    ids, am = _batch()
    out = m(input_ids=ids, attention_mask=am, labels=ids)
    out.loss.backward()
    flat = from_hf_state_dict(mc, m.state_dict(), man).requires_grad_(True)
    lo = oracle_loss(mc, man, flat, ids, attention_mask=am)
    assert abs(float(lo) - float(out.loss)) < 2e-5
    lo.backward()
    tr = Trainer(mc, device="cpu", batch=ids.shape[0], seq=ids.shape[1], init_flat=flat.detach())
    le = tr.loss_and_grad({"input_ids": ids.int(), "attention_mask": am.int(), "labels": ids.int()})
    assert abs(float(le) - float(out.loss)) < 2e-5
    ghf = from_hf_state_dict(mc, {k: (p.grad if p.grad is not None else torch.zeros_like(p))
                                  for k, p in m.named_parameters()}, man)
    assert torch.allclose(flat.grad, ghf, atol=2e-5, rtol=1e-4)
    assert torch.allclose(tr.grad, ghf, atol=2e-5, rtol=1e-4)
    # dropping the scaling gives a measurably different model
    unscaled = dataclasses.replace(mc, rope_scaling=None)
    assert abs(float(oracle_loss(unscaled, man, flat.detach(), ids, attention_mask=am)) - float(out.loss)) > 1e-4


def test_trainer_from_pretrained_llama_directory(tmp_path):
    m = _hf_llama()
    m.save_pretrained(str(tmp_path / "ckpt"))
    tr = Trainer.from_pretrained(str(tmp_path / "ckpt"), device="cpu", batch=2, seq=128)
    assert tr.cfg.vocab_size == VOCAB + 1 and tr.cfg.head_dim == 128  # + [PAD]
    assert dict(tr.cfg.rope_scaling)["rope_type"] == "llama3"
    ids, am = _batch(B=2)
    m.resize_token_embeddings(VOCAB + 1, mean_resizing=False)
    with torch.no_grad():
        m.model.embed_tokens.weight[VOCAB] = m.model.embed_tokens.weight[:VOCAB].mean(0)
    want = m(input_ids=ids, attention_mask=am, labels=ids).loss
    got = tr.eval_loss({"input_ids": ids.int(), "attention_mask": am.int(), "labels": ids.int()})
    assert abs(float(got) - float(want)) < 2e-5
    # an untied checkpoint directory is refused, not loaded as a different model
    m.config.tie_word_embeddings = False
    m.config.save_pretrained(str(tmp_path / "untied"))
    with pytest.raises(ValueError, match="tie_word_embeddings"):
        get_config(str(tmp_path / "untied"))


@pytest.mark.gpu
@pytest.mark.parametrize("T", [64, 256])
def test_engine_on_gpu_matches_hf_llama(T, monkeypatch):
    """The sm_100a engine (bf16, hand-written kernels incl. the head-dim-128 attention and the RoPE table) against
    transformers.LlamaForCausalLM in fp32 on the same device.  T = 64: single-block forward and the GQA backward kernels;
    T = 256: the tiled kernels.  The reference attention is disabled, so a fallback fails the test."""
    assert ops.have_kernels()

    def refuse(*a, **k):
        raise AssertionError("reference attention reached from the engine")
    monkeypatch.setattr(ref, "attention_fwd", refuse)
    monkeypatch.setattr(ref, "attention_bwd", refuse)
    m = _hf_llama(vocab=1003, L=3, seed=3).cuda()
    mc = config_from_hf(m.config.to_dict())
    man = build_manifest(mc)
    B = 8 if T == 64 else 4
    g = torch.Generator().manual_seed(5)
    ids = torch.randint(0, 1002, (B, T), generator=g)
    lens = torch.randint(1, T + 1, (B,), generator=g)
    lens[0] = T
    am = (torch.arange(T)[None] < lens[:, None]).long()
    ids = torch.where(am.bool(), ids, torch.full_like(ids, 1002)).cuda()
    am = am.cuda()
    out = m(input_ids=ids, attention_mask=am, labels=ids)
    out.loss.backward()
    flat = from_hf_state_dict(mc, {k: v.detach().cpu() for k, v in m.state_dict().items()}, man)
    tr = Trainer(mc, device="cuda", batch=B, seq=T, init_flat=flat, use_graph=False)
    assert tr.engine.rope_inv is not None
    loss = tr.loss_and_grad({"input_ids": ids.int(), "attention_mask": am.int(), "labels": ids.int()})
    assert abs(float(loss) - float(out.loss)) < 2e-2, (float(loss), float(out.loss))
    ghf = from_hf_state_dict(mc, {k: (p.grad if p.grad is not None else torch.zeros_like(p)).cpu()
                                  for k, p in m.named_parameters()}, man).cuda()
    cos = torch.nn.functional.cosine_similarity(tr.grad, ghf, dim=0)
    assert float(cos) > 0.995, float(cos)
    for s in man.specs:
        a, b = man.view(tr.grad, s.name).flatten(), man.view(ghf, s.name).flatten()
        if float(b.norm()) > 1e-6:
            assert float(torch.nn.functional.cosine_similarity(a, b, dim=0)) > 0.98, s.name


@pytest.mark.gpu
@pytest.mark.parametrize("inverse", [False, True])
def test_rope_kernel_table_matches_reference(inverse):
    """dtb_rope with an inverse-frequency table (llama3 scaling) against ops.reference.rope_ with the same table."""
    cfg = config_from_hf(_hf_llama().config.to_dict())
    B, T, H, Hkv, hd = 2, 256, 4, 2, cfg.head_dim
    inv = rope_inv_freq(cfg, "cuda")
    torch.manual_seed(4)
    x = torch.randn(B * T, (H + 2 * Hkv) * hd, device="cuda").bfloat16()
    got, want = x.clone(), x.clone()
    ops.rope_(got, B, T, H, Hkv, hd, cfg.rope_theta, inverse=inverse, inv_freq=inv)
    ref.rope_(want, B, T, H, Hkv, hd, cfg.rope_theta, inverse, inv)
    assert (got.float() - want.float()).abs().max().item() < 3e-2
    assert torch.equal(got[:, (H + Hkv) * hd:], x[:, (H + Hkv) * hd:])  # v untouched
    plain = x.clone()
    ref.rope_(plain, B, T, H, Hkv, hd, cfg.rope_theta, inverse)
    assert (plain.float() - want.float()).abs().max().item() > 0.1  # the table really changes the rotation


GOLDEN = os.path.join(os.path.dirname(__file__), "golden", "rope_no_table_hd128.pt")


def rope_golden_input():
    """Seeded input of the no-table RoPE fixture (CPU generator: the same bits everywhere)."""
    g = torch.Generator().manual_seed(11)
    return torch.randn(2 * 64, (4 + 2 * 2) * 128, generator=g).bfloat16()


@pytest.mark.gpu
def test_rope_kernel_without_table_is_unchanged():
    """Without a table the kernel computes theta^(-2i/hd) inline exactly as before the table existed: its output is bitwise
    equal to a fixture written by the table-less kernel (B 2, T 64, H 4, Hkv 2, hd 128, theta 500000, forward + inverse)."""
    want = torch.load(GOLDEN)
    x = rope_golden_input().cuda()
    fwd = x.clone()
    ops.rope_(fwd, 2, 64, 4, 2, 128, 500000.0)
    inv = fwd.clone()
    ops.rope_(inv, 2, 64, 4, 2, 128, 500000.0, inverse=True)
    assert torch.equal(fwd.cpu(), want["forward"])
    assert torch.equal(inv.cpu(), want["inverse"])
