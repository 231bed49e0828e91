"""Causal attention kernel time, head_dim 64 vs 128, against torch SDPA in the same process.

For each shape (tokens, T, H / Hkv, hd): forward and backward time of the tcgen05 kernels (ops.attention_fwd / _bwd on the
packed qkv layout) and of ``torch.nn.functional.scaled_dot_product_attention`` (bf16, ``is_causal``, k / v expanded to H
heads beforehand, backward by ``torch.autograd.grad``), each timed with CUDA events around ``--iters`` back-to-back calls
after ``--warmup`` calls.  Achieved TFLOP/s from shapes: causal forward = 2 * B * H * T^2 * hd (half of the 4 B H T^2 hd of
the two dense products), backward = 2.5 x forward.  At 4096 tokens the operands fit in L2 (warm); at 16384 tokens with
hd 128 they do not.  Prints one JSON line per shape and writes them all to ``--out``.

    python scripts/attn_bench.py --out profiles/attn_hd128_bench.json
"""
import argparse
import json
import math
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch
import torch.nn.functional as F

from distributedtraining_b200 import ops


def card() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    name, power, clock = [s.strip() for s in q[torch.cuda.current_device()].split(",")]
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def timed(fn, warmup: int, iters: int) -> float:
    """Mean milliseconds per call over ``iters`` back-to-back calls (CUDA events)."""
    for _ in range(warmup):
        fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def bench_shape(tokens, T, H, Hkv, hd, warmup, iters):
    B = tokens // T
    M = B * T
    g = torch.Generator(device="cuda").manual_seed(0)
    qkv = (torch.randn(M, (H + 2 * Hkv) * hd, device="cuda", generator=g) * 0.7).bfloat16()
    out = torch.empty(M, H * hd, device="cuda", dtype=torch.bfloat16)
    lse = torch.empty(B, H, T, device="cuda")
    dout = (torch.randn(M, H * hd, device="cuda", generator=g) * 0.5).bfloat16()
    dqkv = torch.empty_like(qkv)
    ours_f = timed(lambda: ops.attention_fwd(qkv, out, lse, B, T, H, hd, Hkv), warmup, iters)
    ours_b = timed(lambda: ops.attention_bwd(dout, qkv, out, lse, dqkv, B, T, H, hd, Hkv), warmup, iters)

    q, k, v = qkv.view(B, T, H + 2 * Hkv, hd).split([H, Hkv, Hkv], dim=2)
    q = q.transpose(1, 2).contiguous().requires_grad_(True)
    k = k.transpose(1, 2).repeat_interleave(H // Hkv, dim=1).contiguous().requires_grad_(True)
    v = v.transpose(1, 2).repeat_interleave(H // Hkv, dim=1).contiguous().requires_grad_(True)
    do = dout.view(B, T, H, hd).transpose(1, 2).contiguous()
    with torch.no_grad():
        sdpa_f = timed(lambda: F.scaled_dot_product_attention(q, k, v, is_causal=True), warmup, iters)
    o = F.scaled_dot_product_attention(q, k, v, is_causal=True)
    sdpa_b = timed(lambda: torch.autograd.grad(o, (q, k, v), do, retain_graph=True), warmup, iters)
    # same inputs, same answer (bf16 tolerance): the comparison is between equivalent computations
    err = (o.detach().transpose(1, 2).reshape(M, H * hd).float() - out.float()).abs().max().item()

    fl_f = 2.0 * B * H * T * T * hd
    fl_b = 2.5 * fl_f
    tf = lambda fl, ms: round(fl / (ms * 1e-3) / 1e12, 1)
    return {"tokens": tokens, "B": B, "T": T, "H": H, "Hkv": Hkv, "hd": hd,
            "fwd_ms": round(ours_f, 4), "bwd_ms": round(ours_b, 4),
            "sdpa_fwd_ms": round(sdpa_f, 4), "sdpa_bwd_ms": round(sdpa_b, 4),
            "fwd_tflops": tf(fl_f, ours_f), "bwd_tflops": tf(fl_b, ours_b),
            "sdpa_fwd_tflops": tf(fl_f, sdpa_f), "sdpa_bwd_tflops": tf(fl_b, sdpa_b),
            "fwd_speedup_vs_sdpa": round(sdpa_f / ours_f, 3), "bwd_speedup_vs_sdpa": round(sdpa_b / ours_b, 3),
            "max_abs_diff_vs_sdpa": round(err, 4)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--tokens", type=int, nargs="+", default=[4096, 16384])
    ap.add_argument("--seq", type=int, nargs="+", default=[64, 512, 2048])
    ap.add_argument("--heads", nargs="+", default=["24/8", "32/8"], help="H/Hkv pairs")
    ap.add_argument("--hd", type=int, nargs="+", default=[64, 128])
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("attn_bench needs a CUDA device")
    assert ops.have_kernels(), "sm_100a kernel library not loaded"
    info = card()
    print(json.dumps(info), flush=True)
    rows = []
    for hd in a.hd:
        for tokens in a.tokens:
            for T in a.seq:
                for hp in a.heads:
                    H, Hkv = map(int, hp.split("/"))
                    r = dict(bench_shape(tokens, T, H, Hkv, hd, a.warmup, a.iters), **info)
                    print(json.dumps(r), flush=True)
                    rows.append(r)
    if a.out:
        with open(a.out, "w") as f:
            json.dump({"card": info, "method": "CUDA events over back-to-back launches; TFLOP/s from shapes (causal fwd "
                       "2*B*H*T^2*hd, bwd 2.5x fwd)", "rows": rows}, f, indent=1)


if __name__ == "__main__":
    main()
