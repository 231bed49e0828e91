"""Head-dim-128 tcgen05 attention kernels vs the fp32 PyTorch reference: forward, LSE, all three input gradients, dropout,
padding mask (x dropout), PAD keys' zero gradient and the folded qkv bias gradient.  The reference attention is disabled
while the op under test runs, so a shape that is not served by a kernel fails instead of comparing the reference with
itself."""
import pytest
import torch

from distributedtraining_b200 import ops
from distributedtraining_b200.ops import reference as ref

pytestmark = pytest.mark.gpu

HD = 128
REF_FWD, REF_BWD = ref.attention_fwd, ref.attention_bwd


@pytest.fixture(autouse=True)
def no_reference_attention(monkeypatch):
    def refuse(*a, **k):
        raise AssertionError("reference attention reached from the op layer at head_dim 128")
    monkeypatch.setattr(ref, "attention_fwd", refuse)
    monkeypatch.setattr(ref, "attention_bwd", refuse)


def _drop(seed, stream):
    rng = ops.DropoutRng("cuda", seed=seed)
    rng.advance()
    return ops.Drop(rng, stream, 0.1)


# T = 32 .. 128: single-block kernels (bwd only for MHA); larger T: tiled kernels.  24 / 8 is Llama-3.2-3B's GQA shape.
@pytest.mark.parametrize("B,T,H,Hkv", [(4, 32, 2, 2), (4, 64, 2, 2), (5, 64, 12, 12), (2, 64, 24, 8), (3, 96, 2, 2),
                                       (2, 128, 3, 3), (3, 192, 2, 1), (2, 256, 2, 2), (1, 512, 4, 2), (2, 512, 24, 8),
                                       (1, 1024, 2, 2), (1, 2048, 3, 1), (2, 2048, 24, 8)])
def test_attention_hd128_fwd_bwd(B, T, H, Hkv):
    torch.manual_seed(0)
    M = B * T
    qkv = (torch.randn(M, (H + 2 * Hkv) * HD, device="cuda") * 0.7).bfloat16()
    out = torch.zeros(M, H * HD, device="cuda", dtype=torch.bfloat16)
    lse = torch.zeros(B, H, T, device="cuda")
    ops.attention_fwd(qkv, out, lse, B, T, H, HD, Hkv)
    r_out = torch.empty(M, H * HD, device="cuda")
    r_lse = torch.empty(B, H, T, device="cuda")
    REF_FWD(qkv, r_out, r_lse, B, T, H, HD, Hkv)
    assert (out.float() - r_out).abs().max().item() < 2e-2 * max(1.0, r_out.abs().max().item())
    assert (lse - r_lse).abs().max().item() < 2e-2
    dout = (torch.randn(M, H * HD, device="cuda") * 0.5).bfloat16()
    dqkv = torch.zeros_like(qkv)
    dbias = torch.zeros((H + 2 * Hkv) * HD, device="cuda")
    ops.attention_bwd(dout, qkv, out, lse, dqkv, B, T, H, HD, Hkv, dbias=dbias)
    # qkv bias gradient (folded into the single-block kernel for MHA with 128 % T == 0, separate colsum otherwise)
    want = dqkv.float().sum(0)
    assert (dbias - want).abs().max().item() < 2e-3 * max(1.0, want.abs().max().item())
    r_dqkv = torch.empty(M, (H + 2 * Hkv) * HD, device="cuda")
    REF_BWD(dout, qkv, r_out.bfloat16(), r_lse, r_dqkv, B, T, H, HD, Hkv)
    parts = [H * HD, Hkv * HD, Hkv * HD]
    for name, a, b in zip(["dq", "dk", "dv"], dqkv.float().split(parts, dim=1), r_dqkv.split(parts, dim=1)):
        rel = (a - b).norm() / (b.norm() + 1e-8)
        assert rel < 3e-2, (name, float(rel))
        assert (a - b).abs().max().item() < 5e-2 * max(1.0, b.abs().max().item()), name


@pytest.mark.parametrize("B,T,H,Hkv", [(4, 64, 2, 2), (3, 32, 2, 2), (2, 64, 6, 2), (2, 256, 2, 2), (1, 512, 6, 2),
                                       (3, 96, 2, 2)])
def test_attention_hd128_dropout_fwd_bwd(B, T, H, Hkv):
    torch.manual_seed(1)
    M = B * T
    drop = _drop(77, 4)
    qkv = (torch.randn(M, (H + 2 * Hkv) * HD, device="cuda") * 0.7).bfloat16()
    out = torch.zeros(M, H * HD, device="cuda", dtype=torch.bfloat16)
    lse = torch.zeros(B, H, T, device="cuda")
    ops.attention_fwd(qkv, out, lse, B, T, H, HD, Hkv, drop=drop)
    r_out, r_lse = torch.empty(M, H * HD, device="cuda"), torch.empty(B, H, T, device="cuda")
    REF_FWD(qkv, r_out, r_lse, B, T, H, HD, Hkv, drop)
    plain = torch.empty(M, H * HD, device="cuda")
    REF_FWD(qkv, plain, None, B, T, H, HD, Hkv)
    assert (plain - r_out).abs().max().item() > 0.05  # the mask really changes the output
    assert (out.float() - r_out).abs().max().item() < 2e-2 * max(1.0, r_out.abs().max().item())
    assert (lse - r_lse).abs().max().item() < 2e-2
    dout = (torch.randn(M, H * HD, device="cuda") * 0.5).bfloat16()
    dqkv = torch.zeros_like(qkv)
    ops.attention_bwd(dout, qkv, out, lse, dqkv, B, T, H, HD, Hkv, drop=drop)
    r_dqkv = torch.empty(M, (H + 2 * Hkv) * HD, device="cuda")
    REF_BWD(dout, qkv, r_out.bfloat16(), r_lse, r_dqkv, B, T, H, HD, Hkv, drop)
    parts = [H * HD, Hkv * HD, Hkv * HD]
    for name, a, b in zip(["dq", "dk", "dv"], dqkv.float().split(parts, dim=1), r_dqkv.split(parts, dim=1)):
        rel = (a - b).norm() / (b.norm() + 1e-8)
        assert rel < 3e-2, (name, float(rel))


@pytest.mark.parametrize("B,T,H,Hkv", [(6, 64, 2, 2), (4, 32, 2, 2), (3, 128, 3, 3), (2, 256, 2, 2), (2, 512, 6, 2),
                                       (3, 96, 3, 1), (1, 1024, 2, 2), (1, 2048, 3, 1)])
@pytest.mark.parametrize("dropout", [False, True])
def test_attention_hd128_padding_mask_fwd_bwd(B, T, H, Hkv, dropout):
    torch.manual_seed(2)
    M = B * T
    kv = torch.randint(1, T + 1, (B,), device="cuda", dtype=torch.int32)
    kv[0] = T          # one full row
    if B > 1:
        kv[1] = 1      # one row with a single real token
    drop = _drop(5, 7) if dropout else None
    qkv = (torch.randn(M, (H + 2 * Hkv) * HD, device="cuda") * 0.7).bfloat16()
    out = torch.zeros(M, H * HD, device="cuda", dtype=torch.bfloat16)
    lse = torch.zeros(B, H, T, device="cuda")
    ops.attention_fwd(qkv, out, lse, B, T, H, HD, Hkv, drop=drop, kv_len=kv)
    r_out, r_lse = torch.empty(M, H * HD, device="cuda"), torch.empty(B, H, T, device="cuda")
    REF_FWD(qkv, r_out, r_lse, B, T, H, HD, Hkv, drop, kv)
    assert (out.float() - r_out).abs().max().item() < 2e-2 * max(1.0, r_out.abs().max().item())
    assert (lse - r_lse).abs().max().item() < 2e-2
    dout = (torch.randn(M, H * HD, device="cuda") * 0.5).bfloat16()
    dqkv = torch.zeros_like(qkv)
    dbias = torch.zeros((H + 2 * Hkv) * HD, device="cuda")
    ops.attention_bwd(dout, qkv, out, lse, dqkv, B, T, H, HD, Hkv, drop=drop, dbias=dbias, kv_len=kv)
    want = dqkv.float().sum(0)
    assert (dbias - want).abs().max().item() < 2e-3 * max(1.0, want.abs().max().item())
    r_dqkv = torch.empty(M, (H + 2 * Hkv) * HD, device="cuda")
    REF_BWD(dout, qkv, r_out.bfloat16(), r_lse, r_dqkv, B, T, H, HD, Hkv, drop, kv)
    parts = [H * HD, Hkv * HD, Hkv * HD]
    for name, a, b in zip(["dq", "dk", "dv"], dqkv.float().split(parts, dim=1), r_dqkv.split(parts, dim=1)):
        rel = (a - b).norm() / (b.norm() + 1e-8)
        assert rel < 3e-2, (name, float(rel))
        assert (a - b).abs().max().item() < 1e-1 * max(1.0, b.abs().max().item()), name
    # keys of PAD positions receive exactly zero gradient
    dk = dqkv.float()[:, H * HD:(H + Hkv) * HD].view(B, T, -1)
    dv = dqkv.float()[:, (H + Hkv) * HD:].view(B, T, -1)
    for b in range(B):
        if int(kv[b]) < T:
            assert float(dk[b, int(kv[b]):].abs().max()) == 0.0
            assert float(dv[b, int(kv[b]):].abs().max()) == 0.0


def test_attention_hd128_library_accepts_and_rejects():
    """The C entry point serves hd 64 and 128 and still refuses other head dims (return code 10)."""
    import ctypes
    import math
    from distributedtraining_b200.ops import _lib
    L = _lib.lib()
    B, T, H = 1, 64, 2
    for hd, want in ((128, 0), (96, 10), (256, 10)):
        qkv = torch.zeros(B * T, 3 * H * hd, device="cuda", dtype=torch.bfloat16)
        out = torch.zeros(B * T, H * hd, device="cuda", dtype=torch.bfloat16)
        lse = torch.zeros(B, H, T, device="cuda")
        rc = L.dtb_attention_fwd(_lib.ptr(qkv), _lib.ptr(out), _lib.ptr(lse), B, T, H, H, hd, qkv.stride(0), out.stride(0),
                                 ctypes.c_float(1.0 / math.sqrt(hd)), _lib.stream_ptr(), None, 0, ctypes.c_float(0.0), None)
        torch.cuda.synchronize()
        assert rc == want, (hd, rc)
