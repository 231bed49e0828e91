"""Kernel time of the fused Qwen3 QK-norm + RoPE (forward with saves, backward) at Qwen3-1.7B attention shapes (16 q / 8 kv
heads of hd 128), with the plain RoPE kernel on the same buffers for comparison.  Bytes moved are the algorithm's minimum
(every q|k element read and written once, the raw copy and rstd written / read once); GB/s is that over the CUDA-event time
of the kernel, against the 7.7 TB/s HBM3e of one B200.  NBUF buffer sets are cycled so that no launch finds its inputs in
the 126 MB L2."""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from distributedtraining_b200 import ops
from distributedtraining_b200.models.transformer import get_config, rope_inv_freq

HBM_TBS = 7.7

ap = argparse.ArgumentParser()
ap.add_argument("--model", default="qwen3-1.7b")
ap.add_argument("--iters", type=int, default=200)
ap.add_argument("--out", default=None)
a = ap.parse_args()
assert ops.have_kernels(), "the sm_100a kernel library is required"
cfg = get_config(a.model)
H, Hkv, hd = cfg.n_head, cfg.kv_heads, cfg.head_dim
nh, W = H + Hkv, cfg.qkv_dim
inv = rope_inv_freq(cfg, "cuda")
qw = (1 + 0.1 * torch.randn(hd, device="cuda")).bfloat16()
kw = (1 + 0.1 * torch.randn(hd, device="cuda")).bfloat16()
dqw, dkw = torch.zeros(hd, device="cuda"), torch.zeros(hd, device="cuda")
results = []
for B, T in ((8, 512), (2, 2048)):
    M = B * T
    nbuf = 6  # 6 x ~76 MB >> 126 MB L2
    qkv = [torch.randn(M, W, device="cuda").bfloat16() for _ in range(nbuf)]
    raw = [torch.empty(M, nh * hd, device="cuda", dtype=torch.bfloat16) for _ in range(nbuf)]
    rstd = [torch.empty(M, nh, device="cuda") for _ in range(nbuf)]
    qk_bytes = M * nh * hd * 2
    runs = {
        "qk_norm_rope_fwd": (lambda i: ops.qk_norm_rope_fwd(qkv[i], B, T, H, Hkv, hd, qw, kw, cfg.eps, inv, raw[i], rstd[i]),
                             3 * qk_bytes + M * nh * 4),  # read q|k, write q|k, write raw; write rstd
        "qk_norm_rope_fwd_eval": (lambda i: ops.qk_norm_rope_fwd(qkv[i], B, T, H, Hkv, hd, qw, kw, cfg.eps, inv),
                                  2 * qk_bytes),
        "qk_norm_rope_bwd": (lambda i: ops.qk_norm_rope_bwd(qkv[i], B, T, H, Hkv, hd, qw, kw, inv, raw[i], rstd[i], dqw, dkw),
                             3 * qk_bytes + M * nh * 4),  # read dy, read raw, write dx; read rstd
        "rope_plain": (lambda i: ops.rope_(qkv[i], B, T, H, Hkv, hd, cfg.rope_theta, inv_freq=inv), 2 * qk_bytes),
    }
    for i in range(nbuf):  # saves for the backward
        ops.qk_norm_rope_fwd(qkv[i], B, T, H, Hkv, hd, qw, kw, cfg.eps, inv, raw[i], rstd[i])
    for name, (fn, nbytes) in runs.items():
        for i in range(2 * nbuf):
            fn(i % nbuf)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(a.iters):
            fn(i % nbuf)
        e1.record()
        torch.cuda.synchronize()
        us = e0.elapsed_time(e1) * 1e3 / a.iters
        r = {"kernel": name, "model": a.model, "B": B, "T": T, "heads": f"{H}/{Hkv}", "hd": hd, "us": us, "bytes": nbytes,
             "GB_s": nbytes / us / 1e3, "share_of_hbm": nbytes / us / 1e6 / HBM_TBS}
        results.append(r)
        print(json.dumps(r), flush=True)
    del qkv, raw, rstd
    torch.cuda.empty_cache()
if a.out:
    with open(a.out, "w") as f:
        json.dump({"device": torch.cuda.get_device_name(), "results": results}, f, indent=1)
