"""Llama-3.2-3B-shaped training with the head-dim-128 attention kernels vs the same engine with the fp32 reference attention.

Same seed, weights and batches in both runs.  Prints the first step's loss and the cosine of the full gradients, then the
losses of ``--steps`` optimizer steps (lr 5e-4 over a pool of four random-token batches, as scripts/step_bench.py does).

    python scripts/attn_traj_check.py 2 2048
"""
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch

from distributedtraining_b200.models.trainer import Trainer
from distributedtraining_b200.ops import attention as A

B, T = int(sys.argv[1]), int(sys.argv[2])
STEPS = 13
kernel_ok = A._kernel_ok


def run(kernels, grad_only=False):
    A._kernel_ok = kernel_ok if kernels else (lambda *a: False)
    torch.manual_seed(0)
    tr = Trainer("llama-3.2-3b", device="cuda", batch=B, seq=T, lr=5e-4, use_graph=False)
    pool = [torch.randint(0, tr.cfg.vocab_size, (B, T), dtype=torch.int32, device="cuda") for _ in range(4)]
    if grad_only:
        out = float(tr.loss_and_grad(pool[0])), tr.grad.clone()
    else:
        out = [float(tr.step(pool[i % 4])) for i in range(STEPS)]
    del tr
    torch.cuda.empty_cache()
    return out


lk, gk = run(True, grad_only=True)
lr_, gr = run(False, grad_only=True)
print(json.dumps({"B": B, "T": T, "loss_kernel": lk, "loss_ref": lr_,
                  "grad_cos": float(torch.nn.functional.cosine_similarity(gk, gr, dim=0)),
                  "rel_norm_diff": float((gk - gr).norm() / gr.norm())}), flush=True)
del gk, gr
torch.cuda.empty_cache()
print(json.dumps({"kernel_losses": run(True)}), flush=True)
print(json.dumps({"ref_losses": run(False)}), flush=True)
