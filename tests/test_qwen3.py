"""Qwen3 (dense, tied head) against ``transformers.Qwen3ForCausalLM``: the decoupled head dim (n_head * head_dim != hidden),
QK-norm (per-head RMSNorm of q and k before RoPE), the config screens, the manifest, import / export, and the fused
QK-norm + RoPE kernel against its reference op."""
import dataclasses
import json
import os
import subprocess
import sys

import pytest
import torch

transformers = pytest.importorskip("transformers")

from distributedtraining_b200 import ops
from distributedtraining_b200.models.trainer import Trainer
from distributedtraining_b200.models.transformer import (ModelConfig, TransformerEngine, build_manifest, config_from_hf,
                                                         from_hf_state_dict, fused_view, get_config, new_model, oracle_loss,
                                                         rope_inv_freq, _rope)
from distributedtraining_b200.ops import reference as ref

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
VOCAB = 300


def _qwen3_config(vocab=VOCAB, d=256, L=2, H=4, Hkv=2, hd=128, ffn=384, npos=256, theta=1e6, **kw):
    from transformers import Qwen3Config
    return Qwen3Config(vocab_size=vocab, hidden_size=d, intermediate_size=ffn, num_hidden_layers=L, num_attention_heads=H,
                       num_key_value_heads=Hkv, head_dim=hd, max_position_embeddings=npos, rms_norm_eps=1e-6,
                       tie_word_embeddings=True, rope_parameters={"rope_type": "default", "rope_theta": theta},
                       attn_implementation="eager", **kw)


def _hf_qwen3(seed=0, **kw):
    """A tiny Qwen3ForCausalLM in fp32 (default: d 256, 4 / 2 heads of hd 128 -> 512 != 256) with randomised 1-D parameters
    (HF ones-inits the RMSNorm weights, q/k norms included: randomise so that layout mistakes cannot hide)."""
    from transformers import Qwen3ForCausalLM
    torch.manual_seed(seed)
    m = Qwen3ForCausalLM(_qwen3_config(**kw)).eval()
    with torch.no_grad():
        for n, p in m.named_parameters():
            if p.dim() == 1:
                p.add_(0.1 * torch.randn_like(p))
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


# ---------------------------------------------------------------------------------------------------------------------
# config, manifest
# ---------------------------------------------------------------------------------------------------------------------
def test_config_layouts_and_screens():
    d5 = _qwen3_config().to_dict()
    assert d5["model_type"] == "qwen3"
    c5, c4 = config_from_hf(d5), config_from_hf(_legacy(d5))
    assert c5 == c4
    assert c5.family == "llama" and c5.qk_norm and c5.head_dim == 128 and c5.n_head * c5.head_dim != c5.n_embd
    assert (c5.kv_heads, c5.rope_theta, c5.rope_scaling, c5.eps) == (2, 1e6, None, 1e-6)
    assert c5.qkv_dim == (4 + 2 * 2) * 128
    # head_dim absent: hidden / heads
    assert config_from_hf({k: v for k, v in d5.items() if k != "head_dim"}).head_dim == 256 // 4
    # every unsupported feature is refused with the field named
    for field, val in (("tie_word_embeddings", False), ("attention_bias", True), ("use_sliding_window", True),
                       ("hidden_act", "gelu")):
        with pytest.raises(ValueError, match=field):
            config_from_hf(dict(d5, **{field: val}))
    with pytest.raises(ValueError, match="tie_word_embeddings"):
        config_from_hf({k: v for k, v in d5.items() if k != "tie_word_embeddings"})  # Qwen3Config's default is untied
    with pytest.raises(ValueError, match="layer_types"):
        config_from_hf(dict(d5, layer_types=["full_attention", "sliding_attention"]))
    yarn = {"rope_type": "yarn", "factor": 4.0, "original_max_position_embeddings": 32768}
    with pytest.raises(ValueError, match="yarn"):
        config_from_hf(dict(d5, rope_parameters=dict(yarn, rope_theta=1e6)))
    with pytest.raises(ValueError, match="yarn"):
        config_from_hf(dict(_legacy(d5), rope_scaling=yarn))
    # the Llama screen of a decoupled head dim is unchanged
    from transformers import LlamaConfig
    ld = LlamaConfig(hidden_size=256, num_attention_heads=4, tie_word_embeddings=True).to_dict()
    with pytest.raises(ValueError, match="head_dim"):
        config_from_hf(dict(ld, head_dim=128))
    # presets
    for name, (d, L, H) in {"qwen3-0.6b": (1024, 28, 16), "qwen3-1.7b": (2048, 28, 16), "qwen3-4b": (2560, 36, 32)}.items():
        c = get_config(name)
        assert (c.n_embd, c.n_layer, c.n_head, c.kv_heads, c.head_dim) == (d, L, H, 8, 128)
        assert (c.vocab_size, c.rope_theta, c.eps, c.n_positions, c.rope_scaling, c.qk_norm) == (151936, 1e6, 1e-6, 40960, None, True)
    t = get_config("qwen3-tiny")
    assert (t.vocab_size, t.n_embd, t.n_head, t.head_dim, t.kv_heads, t.ffn_dim, t.n_layer) == (512, 128, 4, 64, 2, 256, 2)
    assert t.n_head * t.head_dim != t.n_embd
    # the new fields leave the existing configs as they were
    assert ModelConfig().head_dim == 64 and not ModelConfig().qk_norm
    assert get_config("llama-3.2-3b").head_dim == 128 and get_config("llama-3.2-1b").head_dim == 64


@pytest.mark.parametrize("name,n_params,n_tensors", [("qwen3-0.6b", 596049920, 310), ("qwen3-1.7b", 1720574976, 310),
                                                     ("qwen3-4b", 4022468096, 398)])
def test_manifest_matches_hf_meta_model(name, n_params, n_tensors):
    from transformers import Qwen3ForCausalLM
    c = get_config(name)
    hc = _qwen3_config(vocab=c.vocab_size, d=c.n_embd, L=c.n_layer, H=c.n_head, Hkv=c.kv_heads, hd=c.head_dim, ffn=c.ffn_dim,
                       npos=c.n_positions)
    with torch.device("meta"):
        m = Qwen3ForCausalLM(hc)
    hf = dict(m.named_parameters())  # the tied head is one parameter
    man = build_manifest(c)
    assert man.num_params == sum(p.numel() for p in hf.values()) == n_params
    assert len(man) == len(hf) == n_tensors
    assert man.same_layout({k: tuple(p.shape) for k, p in hf.items()})
    assert dataclasses.replace(config_from_hf(hc.to_dict()), name=c.name) == c
    # q_norm / k_norm sit between v_proj and o_proj: q|k|v stays one fused view and the arena stays in program order
    names = man.names
    for l in range(c.n_layer):
        p = f"model.layers.{l}.self_attn."
        i = names.index(p + "v_proj.weight")
        assert names[i + 1:i + 4] == [p + "q_norm.weight", p + "k_norm.weight", p + "o_proj.weight"]
        assert man[p + "q_norm.weight"].shape == (128,) and man[p + "q_norm.weight"].init == "ones"
    flat = torch.zeros(man.total, device="meta")
    assert tuple(fused_view(man, flat, [f"model.layers.0.self_attn.{x}_proj.weight" for x in "qkv"]).shape) == (c.qkv_dim, c.n_embd)


# ---------------------------------------------------------------------------------------------------------------------
# reference op, parity with transformers (CPU, fp32)
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("hd", [64, 128])
def test_reference_op_backward_matches_autograd(hd):
    B, T, H, Hkv = 2, 16, 4, 2
    nh = H + Hkv
    torch.manual_seed(0)
    cfg = ModelConfig(family="llama", n_embd=128, n_head=H, n_kv_head=Hkv, n_head_dim=hd, rope_theta=1e6, qk_norm=True)
    inv = rope_inv_freq(cfg)
    x = torch.randn(B * T, (H + 2 * Hkv) * hd, dtype=torch.float64).float()
    qw, kw = 1 + 0.2 * torch.randn(hd), 1 + 0.2 * torch.randn(hd)
    dy = torch.randn_like(x)
    xa, qa, ka = x.clone().requires_grad_(True), qw.clone().requires_grad_(True), kw.clone().requires_grad_(True)
    # autograd of the oracle's formulation: per-head RMSNorm, then _rope
    x4 = xa.view(B, T, H + 2 * Hkv, hd)
    q, k, v = x4[:, :, :H], x4[:, :, H:nh], x4[:, :, nh:]
    q = _rope(q * torch.rsqrt(q.pow(2).mean(-1, keepdim=True) + 1e-6) * qa, inv)
    k = _rope(k * torch.rsqrt(k.pow(2).mean(-1, keepdim=True) + 1e-6) * ka, inv)
    y = torch.cat([q, k, v], dim=2).reshape(B * T, -1)
    (y * dy).sum().backward()
    out, raw, rstd = x.clone(), torch.empty(B * T, nh * hd), torch.empty(B * T, nh)
    ref.qk_norm_rope_fwd(out, B, T, H, Hkv, hd, qw, kw, 1e-6, inv, raw, rstd)
    assert torch.allclose(out, y.detach()) and torch.equal(raw, x[:, :nh * hd])
    assert torch.equal(out[:, nh * hd:], x[:, nh * hd:])  # v untouched
    d = dy.clone()
    dq, dk = torch.ones(hd), torch.ones(hd)  # accumulated into
    ref.qk_norm_rope_bwd(d, B, T, H, Hkv, hd, qw, kw, inv, raw, rstd, dq, dk)
    assert torch.allclose(d[:, :nh * hd], xa.grad[:, :nh * hd], atol=1e-5, rtol=1e-4)
    assert torch.equal(d[:, nh * hd:], dy[:, nh * hd:])
    assert torch.allclose(dq - 1, qa.grad, atol=1e-4, rtol=1e-4) and torch.allclose(dk - 1, ka.grad, atol=1e-4, rtol=1e-4)


@pytest.mark.parametrize("layout", ["v5", "v4"])
def test_loss_and_grads_match_hf_qwen3(layout):
    m = _hf_qwen3()
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
    assert float(man.view(ghf, "model.layers.0.self_attn.q_norm.weight").norm()) > 0
    assert torch.allclose(flat.grad, ghf, atol=2e-5, rtol=1e-4)
    assert torch.allclose(tr.grad, ghf, atol=2e-5, rtol=1e-4)
    # without QK-norm it is measurably a different model
    plain = dataclasses.replace(mc, qk_norm=False)
    pman = build_manifest(plain)
    pflat = torch.zeros(pman.total)
    for s in pman:
        pman.view(pflat, s.name).copy_(man.view(flat.detach(), s.name))
    assert abs(float(oracle_loss(plain, pman, pflat, ids, attention_mask=am)) - float(out.loss)) > 1e-4


def test_trainer_from_pretrained_and_strict_export(tmp_path):
    from transformers import Qwen3ForCausalLM
    m = _hf_qwen3()
    m.save_pretrained(str(tmp_path / "ckpt"))
    tr = Trainer.from_pretrained(str(tmp_path / "ckpt"), device="cpu", batch=2, seq=128)
    assert tr.cfg.vocab_size == VOCAB + 1 and tr.cfg.head_dim == 128 and tr.cfg.qk_norm  # + [PAD]
    ids, am = _batch(B=2)
    m.resize_token_embeddings(VOCAB + 1, mean_resizing=False)
    with torch.no_grad():
        m.model.embed_tokens.weight[VOCAB] = m.model.embed_tokens.weight[:VOCAB].mean(0)
    want = m(input_ids=ids, attention_mask=am, labels=ids)
    got = tr.eval_loss({"input_ids": ids.int(), "attention_mask": am.int(), "labels": ids.int()})
    assert abs(float(got) - float(want.loss)) < 2e-5
    # export (the averaged_model.pt format) loads strictly into Qwen3ForCausalLM and gives the same logits
    back = Qwen3ForCausalLM(_qwen3_config(vocab=VOCAB + 1)).eval()
    back.load_state_dict(tr.hf_state_dict(), strict=True)
    with torch.no_grad():
        assert torch.allclose(back(input_ids=ids, attention_mask=am).logits, want.logits, atol=1e-5, rtol=1e-5)
    # an untied checkpoint directory is refused, not loaded as a different model
    m.config.tie_word_embeddings = False
    m.config.save_pretrained(str(tmp_path / "untied"))
    with pytest.raises(ValueError, match="tie_word_embeddings"):
        get_config(str(tmp_path / "untied"))


def test_fused_delta_and_peer_source_forward_qwen3():
    """dual-B (x (W+dW)^T without materialising W+dW) and persist-B (weights read from a source arena) give the loss of the
    materialised model; the q/k norm weights are small tensors (base+delta in the arena, read from the source)."""
    torch.manual_seed(0)
    cfg, man, arena = new_model("qwen3-tiny")
    base = arena.flat.clone()
    delta = torch.randn_like(base) * 0.01
    B, T = 2, 16
    ids = torch.randint(0, cfg.vocab_size, (B, T), dtype=torch.int32)
    eng = TransformerEngine(cfg, man, (base + delta).clone(), None, B, T, lm_chunk=32)
    eng.set_batch(ids)
    want = float(eng.forward_loss())
    p = base.clone()
    eng2 = TransformerEngine(cfg, man, p, None, B, T, lm_chunk=16)
    small = set(eng2.small_chunk_ids().tolist())
    _, _, ct = man.seg_table("cpu")
    for n in ("model.layers.1.self_attn.q_norm.weight", "model.layers.1.self_attn.k_norm.weight"):
        assert any(int(ct[c]) == man.index(n) for c in small), n
    ops.weighted_avg(base, [delta], torch.ones(1, len(man)), man, [p], chunk_ids=eng2.small_chunk_ids(), unit_base=True)
    eng2.set_delta(delta)
    eng2.set_batch(ids)
    assert abs(float(eng2.forward_loss()) - want) < 1e-5
    local = torch.zeros_like(base)
    eng3 = TransformerEngine(cfg, man, local, None, B, T, lm_chunk=16)
    eng3.set_source((base + delta).clone())
    eng3.set_batch(ids)
    assert abs(float(eng3.forward_loss()) - want) < 1e-5
    eng3.persist_small_from_source()
    eng3.set_source(None)
    for sp in man:
        assert torch.allclose(man.view(local, sp.name), man.view(base + delta, sp.name)), sp.name
    assert abs(float(eng3.forward_loss()) - want) < 1e-5


def test_two_miners_one_averager_qwen3_tiny(tmp_path):
    from transformers import Qwen3ForCausalLM
    args = ["--roles", "miner:0-1,averager:2", "--device", "cpu", "--backend", "disk", "--model", "qwen3-tiny", "--batch_size", "4",
            "--seq_len", "16", "--local_steps", "5", "--rounds", "2", "--meta_epochs", "1", "--storage.model_dir", str(tmp_path / "model"),
            "--storage.gradient_dir", str(tmp_path / "grad"), "--metrics_jsonl", str(tmp_path / "metrics.jsonl")]
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=3", "--master-addr", "127.0.0.1",
           "--master-port", "29651", os.path.join(ROOT, "neurons", "run.py")] + args
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=420, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-3000:]
    for rk in (0, 1):
        assert int(open(tmp_path / "model" / "deltas" / f"weight_diff_{rk}.pt.round").read()) == 2
    assert int(open(tmp_path / "model" / "base" / "averaged_model.pt.round").read()) >= 1
    sd = torch.load(tmp_path / "model" / "averaged_model.pt", weights_only=False)
    assert len(sd) == 2 * 11 + 2 + 1 and all(torch.isfinite(v).all() for v in sd.values())
    c = get_config("qwen3-tiny")
    m = Qwen3ForCausalLM(_qwen3_config(vocab=c.vocab_size, d=c.n_embd, L=c.n_layer, H=c.n_head, Hkv=c.kv_heads, hd=c.head_dim,
                                       ffn=c.ffn_dim, npos=c.n_positions))
    m.load_state_dict(sd, strict=True)
    recs = [json.loads(l) for l in open(tmp_path / "metrics.jsonl")]
    assert any(r.get("role") == "averager" and "loss_averaged" in r for r in recs)
    assert any(r.get("role") == "miner" and "train_loss" in r for r in recs)


# ---------------------------------------------------------------------------------------------------------------------
# GPU: the fused kernel, the engine against transformers, CUDA graphs
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("T", [64, 256])
@pytest.mark.parametrize("H,Hkv", [(4, 2), (16, 8)])
@pytest.mark.parametrize("hd", [64, 128])
def test_qk_norm_rope_kernel_matches_reference(hd, H, Hkv, T):
    assert ops.have_kernels()
    B, nh = 2, H + Hkv
    M, W = B * T, (H + 2 * Hkv) * hd
    cfg = ModelConfig(family="llama", n_embd=128, n_head=H, n_kv_head=Hkv, n_head_dim=hd, rope_theta=1e6, qk_norm=True)
    inv = rope_inv_freq(cfg, "cuda")
    g = torch.Generator(device="cuda").manual_seed(hd + H + T)
    x = (3 * torch.randn(M, W, device="cuda", generator=g)).bfloat16()
    qw = (1 + 0.3 * torch.randn(hd, device="cuda", generator=g)).bfloat16()
    kw = (1 + 0.3 * torch.randn(hd, device="cuda", generator=g)).bfloat16()
    # forward
    got, raw, rstd = x.clone(), torch.empty(M, nh * hd, device="cuda", dtype=torch.bfloat16), torch.empty(M, nh, device="cuda")
    ops.qk_norm_rope_fwd(got, B, T, H, Hkv, hd, qw, kw, 1e-6, inv, raw, rstd)
    want, rraw, rrstd = x.clone(), torch.empty_like(raw), torch.empty_like(rstd)
    ref.qk_norm_rope_fwd(want, B, T, H, Hkv, hd, qw, kw, 1e-6, inv, rraw, rrstd)
    assert torch.equal(got[:, nh * hd:], x[:, nh * hd:])  # v bitwise untouched
    assert torch.equal(raw, x[:, :nh * hd])
    assert torch.allclose(rstd, rrstd, rtol=1e-5, atol=0)
    assert (got.float() - want.float()).abs().max().item() < 4e-2  # |y| ~ |w| <= 2.5: a few bf16 ulps
    # eval form (no saves) writes the same output
    ev = x.clone()
    ops.qk_norm_rope_fwd(ev, B, T, H, Hkv, hd, qw, kw, 1e-6, inv)
    assert torch.equal(ev, got)
    # backward: kernel vs the fp32 reference on the same saves
    dy = torch.randn(M, W, device="cuda", generator=g).bfloat16()
    dq0 = torch.randn(hd, device="cuda", generator=g)
    dk0 = torch.randn(hd, device="cuda", generator=g)
    dgot, dq, dk = dy.clone(), dq0.clone(), dk0.clone()
    ops.qk_norm_rope_bwd(dgot, B, T, H, Hkv, hd, qw, kw, inv, raw, rstd, dq, dk)
    dwant, rq, rk = dy.float(), dq0.clone(), dk0.clone()
    ref.qk_norm_rope_bwd(dwant, B, T, H, Hkv, hd, qw.float(), kw.float(), inv, raw.float(), rstd, rq, rk)
    assert torch.equal(dgot[:, nh * hd:], dy[:, nh * hd:])
    err = (dgot.float() - dwant)[:, :nh * hd]
    assert err.abs().max().item() < 2e-2 * dwant[:, :nh * hd].abs().max().item() + 1e-3
    for a, b, b0 in ((dq, rq, dq0), (dk, rk, dk0)):
        assert ((a - b).norm() / (b - b0).norm()).item() < 1e-2


def _refuse_reference(monkeypatch):
    def refuse(*a, **k):
        raise AssertionError("reference op reached from the engine")
    for name in ("attention_fwd", "attention_bwd", "qk_norm_rope_fwd", "qk_norm_rope_bwd"):
        monkeypatch.setattr(ref, name, refuse)


@pytest.mark.gpu
@pytest.mark.parametrize("T", [64, 256])
def test_engine_on_gpu_matches_hf_qwen3(T, monkeypatch):
    """The sm_100a engine (bf16; fused QK-norm + RoPE, hd-128 GQA attention) against Qwen3ForCausalLM in fp32 on the same
    device.  T = 64: single-block attention; T = 256: the tiled kernels.  The reference attention and QK-norm are refused."""
    assert ops.have_kernels()
    _refuse_reference(monkeypatch)
    m = _hf_qwen3(vocab=1003, L=3, seed=3).cuda()
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
    loss = tr.loss_and_grad({"input_ids": ids.int(), "attention_mask": am.int(), "labels": ids.int()})
    assert abs(float(loss) - float(out.loss)) < 2e-2, (float(loss), float(out.loss))
    ghf = from_hf_state_dict(mc, {k: (p.grad if p.grad is not None else torch.zeros_like(p)).cpu()
                                  for k, p in m.named_parameters()}, man).cuda()
    cos = torch.nn.functional.cosine_similarity(tr.grad, ghf, dim=0)
    assert float(cos) > 0.995, float(cos)
    checked = set()
    for s in man.specs:
        a, b = man.view(tr.grad, s.name).flatten(), man.view(ghf, s.name).flatten()
        if float(b.norm()) > 1e-6:
            assert float(torch.nn.functional.cosine_similarity(a, b, dim=0)) > 0.98, s.name
            checked.add(s.name.split(".")[-2])
    assert {"q_norm", "k_norm"} <= checked


@pytest.mark.gpu
def test_graph_step_equals_eager_and_learns(monkeypatch):
    assert ops.have_kernels()
    _refuse_reference(monkeypatch)
    B, T = 8, 64
    g = torch.Generator(device="cuda").manual_seed(0)
    pool = [torch.randint(0, 512, (B, T), dtype=torch.int32, device="cuda", generator=g) for _ in range(2)]
    runs = {}
    for graph in (False, True):
        tr = Trainer("qwen3-tiny", device="cuda", batch=B, seq=T, lr=2e-3, use_graph=graph)
        runs[graph] = ([float(tr.step(pool[i % 2])) for i in range(12)], tr.master.clone())
    (le, me), (lg, mg) = runs[False], runs[True]
    assert max(abs(a - b) for a, b in zip(le, lg)) < 2e-2, (le, lg)
    assert float(torch.nn.functional.cosine_similarity(me - tr.base, mg - tr.base, dim=0)) > 0.99
    assert lg[-1] < lg[0] - 0.5, lg
