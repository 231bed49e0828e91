#!/usr/bin/env python
"""Headline benchmark (driver contract): local-SGD / delta-averaging training of GPT-2-small on N B200 GPUs of one node.

Metric (BASELINE.json): tokens/sec (whole job; per-miner = value / N) and avg-round wall-time, device-timed, max over
ranks, GPT-2-small (124.4 M params, vocab 50258), bf16 compute, N miners, ``local_steps`` optimizer steps per round
followed by the fused delta all-gather -> weighted-average -> base broadcast (+ ``meta_steps`` learned-mixer steps).

    python bench.py --gpus 1 --steps 50 --warmup 5
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 --master-port 29500 \
        bench.py --gpus 8 --steps 50 --warmup 5
    python bench.py --impl reference ...      # the reference arm (see baseline/reference_arm.py)

Two timed regions of exactly K steps each (both bracketed by barrier + cuda synchronize, CUDA events, max over ranks):
  * ``value``: inputs already resident on the device (kernel/collective time only);
  * ``e2e``:   through the public API (``training_manager.DeltaLoop.train``): every step copies its input batch from
               pinned host memory and copies the step's loss back to pinned host memory.
Every timed region performs at least one averaging round (with ``--meta-steps`` learned-mixer steps).  A third region
(``full_round``) measures ONE WHOLE ROUND directly: ``--local-steps`` optimizer steps + the reference-faithful learned mixer
(``--meta-epochs``^2 passes over ``--val-texts`` sequences @ ``--val-seq``, run by all ranks) + averaging + base broadcast.
Data: synthetic tokens; weights: random init.  ``--impl reference`` = the unmodified upstream miner, ``--impl torch-bf16`` = HF
GPT-2 under bf16 autocast + SDPA + fused AdamW + NCCL round (the strongest stock-library baseline).

``--dump-outputs DIR`` writes what the ``value`` region computed, as float32 ``.npy`` files (rank 0): ``loss`` (the mean loss
of its last step), ``theta_sample`` (a fixed, seeded sample of the fp32 weights the next step starts from) and ``mixer_w``
(the mixing weights [miners, tensors] of its last round).  Inputs and initial weights are seeded, so two builds run with the
same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)


def parse_args(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", type=str, default="ours", choices=["ours", "reference", "nccl", "nvls", "torch-bf16"])
    ap.add_argument("--model", type=str, default="gpt2")
    ap.add_argument("--batch-size", type=int, default=512, help="sequences per miner per step (both arms use the same default)")
    ap.add_argument("--seq-len", type=int, default=64, help="reference miner sequence length (neurons/miner.py:70)")
    ap.add_argument("--local-steps", type=int, default=100)
    ap.add_argument("--meta-steps", type=int, default=1, help="learned-mixer SGD steps in the rounds of the K-step timed regions")
    ap.add_argument("--meta-epochs", type=int, default=7, help="full-round region: meta_epochs^2 passes over the validation set "
                    "(reference neurons/averager.py:106: 7)")
    ap.add_argument("--val-texts", type=int, default=100, help="validation sequences (reference neurons/averager.py:61)")
    ap.add_argument("--val-seq", type=int, default=512, help="validation sequence length (reference neurons/averager.py:72)")
    ap.add_argument("--val-batch", type=int, default=8, help="averager batch size (reference: --batch_size; validator uses 8)")
    ap.add_argument("--meta-mode", type=str, default="auto", choices=["auto", "replicate", "dp"])
    ap.add_argument("--no-full-round", action="store_true", help="skip the directly measured whole round (100 local steps + "
                    "reference-faithful meta-learning + averaging)")
    ap.add_argument("--delta-dtype", type=str, default="fp32", choices=["fp32", "bf16", "fp8"])
    ap.add_argument("--lr", type=float, default=5e-4)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--dropout", type=float, default=None, help="train-mode dropout; default = the model preset (GPT-2: 0.1, as in the reference)")
    ap.add_argument("--fp8-forward", action="store_true", help="e4m3 forward GEMMs with delayed scaling (config 4)")
    ap.add_argument("--fp8-backward", action="store_true", help="with --fp8-forward: fp8 dgrad GEMMs (e5m2 gradients x transposed e4m3 weights)")
    ap.add_argument("--dump-outputs", type=str, default=None, metavar="DIR",
                    help="write the loss, weights (seeded sample) and mixing weights of the timed steps to DIR/<name>.npy")
    return ap.parse_args(argv)


def shared_config(model_desc: str, B: int, T: int, world: int) -> dict:
    """``config`` block emitted IDENTICALLY by every arm (ours / reference / torch-bf16 / nccl): what is being measured.
    Arm-specific details live in the top-level ``detail`` key."""
    return {"model": model_desc, "global_batch": B * world, "micro_batch_per_miner": B, "seq_len": T,
            "parallelism": f"dp{world} (one miner per GPU, local-SGD delta averaging)",
            "l2_policy": "per-step working set (>= 2 GB of weights, optimizer state and activations) >> 126 MB L2"}


GPT2_SMALL_DESC = "gpt2-small + [PAD] (124440576 params, vocab 50258)"
DUMP_THETA_SAMPLE = 1 << 22  # fp32 weights kept by --dump-outputs: 16 MB, whatever the model size


def capture_outputs(trainer, coord) -> dict:
    """Host copies of what a caller of the timed steps holds after the last one: that step's loss, the weights the next
    step starts from (a fixed, seeded sample) and the mixing weights.  Reads only: the trainer's state is left as it is."""
    import torch

    coord.sync_base()  # a base pushed by the peers must have landed before it is read
    theta = trainer.base if trainer.master_stale else trainer.master  # right after a round theta lives in theta_base
    n = theta.numel()
    if n <= DUMP_THETA_SAMPLE:
        idx = torch.arange(n)
    else:
        idx = torch.randint(n, (DUMP_THETA_SAMPLE,), generator=torch.Generator().manual_seed(0)).sort().values
    out = {"loss": trainer.engine.loss.reshape(1),  # the device buffer Trainer.step returns
           "theta_sample": theta[idx.to(theta.device)], "mixer_w": coord.w}
    return {k: v.detach().float().cpu().numpy() for k, v in out.items()}


def write_outputs(out_dir: str, arrays: dict) -> None:
    import numpy as np

    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


# ---------------------------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi sampler running DURING the timed region (B200_PROFILING.md clocks line)."""

    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown," \
        "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index: int):
        self.gpu_index = gpu_index
        self.proc = None
        self.path = None

    def start(self):
        try:
            f = tempfile.NamedTemporaryFile("w", suffix=".csv", delete=False)
            self.path = f.name
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.gpu_index)], stdout=f, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.12)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, power = [], [], set(), []
        try:
            for line in open(self.path):
                p = [x.strip() for x in line.split(",")]
                if len(p) < 9:
                    continue
                try:
                    sm.append(float(p[1])); mx.append(float(p[2])); power.append(float(p[3]))
                except ValueError:
                    continue
                for name, val in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], p[5:9]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


def maybe_respawn(args) -> None:
    """``python bench.py --gpus N`` without torchrun: re-launch ourselves under torch.distributed.run."""
    if args.gpus > 1 and "RANK" not in os.environ:
        port = 29500 + (os.getpid() % 2000)
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", str(port), os.path.abspath(__file__)] + sys.argv[1:]
        raise SystemExit(subprocess.call(cmd))


# ---------------------------------------------------------------------------------------------------------------------
def run_ours(args) -> dict:
    import torch
    import torch.distributed as dist

    from distributedtraining_b200 import ops
    from distributedtraining_b200.data import SyntheticTokens
    from distributedtraining_b200.models.trainer import Trainer
    from distributedtraining_b200.parallel.exchange import CollectiveExchange, PeerExchange
    from distributedtraining_b200.parallel.launch import barrier_sync, init_distributed, max_over_ranks
    from distributedtraining_b200.parallel.local_sgd import LocalSGDCoordinator
    from distributedtraining_b200.training_manager import DeltaLoop

    rank, world, device = init_distributed("nccl")
    assert device.type == "cuda", "bench.py needs a GPU"
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world}"
    B, T, K, W = args.batch_size, args.seq_len, args.steps, args.warmup
    from distributedtraining_b200.models.transformer import build_manifest, get_config
    man = build_manifest(get_config(args.model))
    buffers = None
    if args.impl == "nccl":
        ex = CollectiveExchange(man, delta_dtype=args.delta_dtype) if world > 1 else None
        plane = "nccl all_gather / all_reduce + torch" if world > 1 else "local torch"
    elif args.impl == "nvls" and world > 1:
        from distributedtraining_b200.parallel.exchange import NvlsExchange
        ex = NvlsExchange(man)  # uniform mixer: in-switch reduction + multicast of the new base
        plane = "NVLS (multimem.ld_reduce + multimem.st), uniform mixer"
        args.meta_steps = 0
    else:
        # the windows come first: the trainer's theta_base and bf16 compute copy LIVE in them, so that the peers' averaging
        # kernels can land the new base there directly (multimem.st through the NVSwitch when the windows are multicast-bound)
        ex = PeerExchange(man, delta_dtype=args.delta_dtype)
        buffers = ex.trainer_buffers()
        plane = f"peer windows ({ex.win.backing}, multicast={'yes' if ex.win.mc_ptr else 'no'}): sharded fused averaging kernels, no NCCL"
    # seed=0: the same theta_base on every rank; dropout_seed=rank: independent dropout masks per miner
    trainer = Trainer(args.model, device=device, batch=B, seq=T, lr=args.lr, seed=0, dropout_seed=rank,
                      fp8_forward=args.fp8_forward, fp8_backward=args.fp8_backward, dropout=args.dropout, buffers=buffers)
    V = trainer.cfg.vocab_size
    dev_data = SyntheticTokens(B, T, V, seed=1000 + rank, device=str(device), pool=8)
    host_data = SyntheticTokens(B, T, V, seed=2000 + rank, pool=8, pin=True)
    # validation set of the averager: ``val_texts`` sequences @ ``val_seq`` in batches of ``val_batch`` (the last one smaller),
    # identical on every rank (reference neurons/averager.py:58-94)
    Tv = min(args.val_seq, trainer.cfg.n_positions)
    Bv = min(args.val_batch, args.val_texts)
    vs = SyntheticTokens(args.val_texts, Tv, V, seed=7, device=str(device), pool=1).pool[0]
    val = [{k: v[i:i + Bv] for k, v in vs.items()} for i in range(0, args.val_texts, Bv)]
    learned = args.impl != "nvls"
    coord = LocalSGDCoordinator(trainer, ex, meta_steps=args.meta_steps, mixer="learned" if learned else "uniform",
                                val_batches=val, post_pull_lr=5e-5, meta_mode=args.meta_mode)
    # the optimizer keeps lr=5e-4 in round 0 and 5e-5 after the first pull, as in the reference miner

    def run_steps(n: int, pool, gstep0: int, force_round: bool) -> int:
        g = gstep0
        did_round = False
        for i in range(n):
            trainer.step(pool[i % len(pool)])  # dict batch: input_ids + kv_len (padding mask); labels = input_ids
            g += 1
            if g % args.local_steps == 0:
                coord.finish_round()
                did_round = True
        if force_round and not did_round:
            coord.finish_round()
        return g

    # ---- warm-up (includes graph capture and one averaging round) ----
    g = run_steps(max(W, 3), dev_data.pool, 0, force_round=True)
    trainer.step(dev_data.pool[0])  # the first step after a round has its own graph (in-GEMM flag acquires): capture it untimed too
    barrier_sync(device)
    coord.timer.summary()  # drop the warm-up round's phase events

    # ---- region 1: device-resident inputs ----
    sampler = ClockSampler(device.index)
    sampler.start()
    c0 = ops.launch_count()
    rounds0 = coord.round
    barrier_sync(device)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    g = run_steps(K, dev_data.pool, 0, force_round=True)
    e1.record()
    barrier_sync(device)
    clocks = sampler.stop()
    ms_total = max_over_ranks(e0.elapsed_time(e1), device)
    phases = coord.timer.summary()
    rounds = coord.round - rounds0
    eager_launches = ops.launch_count() - c0
    outputs = capture_outputs(trainer, coord) if args.dump_outputs and rank == 0 else None
    launches = K * trainer.launches_per_step + (eager_launches if trainer.use_graph else eager_launches - K * trainer.launches_per_step)
    tokens = K * B * T * world
    desc = GPT2_SMALL_DESC if trainer.cfg.name == "gpt2" else f"{trainer.cfg.name} ({trainer.man.num_params} params, vocab {V})"
    result = {
        "metric": f"tokens/sec ({'GPT-2-small' if trainer.cfg.name == 'gpt2' else trainer.cfg.name} local-SGD training, all miners; per-miner = value / n_gpus)",
        "value": tokens / ms_total * 1e3, "unit": "tokens/s", "n_gpus": world, "steps": K, "warmup": max(W, 3),
        "ms_per_step": ms_total / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
        "data": "synthetic tokens (Zipf ids, right-padded), random-init weights", "impl": args.impl,
        "tokens_per_s_per_miner": tokens / ms_total * 1e3 / world, "rounds_in_timed_region": rounds,
        "config": shared_config(desc, B, T, world),
        "detail": {"local_steps": args.local_steps, "meta_steps_in_timed_rounds": coord.meta_steps, "delta_dtype": args.delta_dtype,
                   "exchange": plane, "optimizer": "fused AdamW (fp32 master, bf16 compute)", "fp8_forward": bool(args.fp8_forward), "fp8_dgrad": bool(args.fp8_backward and args.fp8_forward),
                   "dropout": trainer.cfg.dropout, "padding_mask": "attention_mask -> kv_len in the attention kernels",
                   "cuda_graph": bool(trainer.use_graph), "base_broadcast": getattr(coord, "last_round_mode", None),
                   "first_forward_after_round": "forward GEMMs acquire the shard owners' base flags in-kernel (no wait kernel)"
                   if coord.fused_first_forward else "wait kernel / pull pass before the step",
                   "meta": coord.meta.describe() if coord.meta is not None else None},
        "clocks": clocks, "gpu_launches": int(launches),
        "round_phase_ms_rank0": {k: round(v / max(rounds, 1), 3) for k, v in phases.items()},
    }
    # ---- region 2: end to end through the public API (pinned-host inputs, per-step loss read-back) ----
    if not args.no_e2e:
        loop = DeltaLoop(device, args.model, host_data, learning_rate=args.lr, hf_manager=None, trainer=trainer,
                         local_steps=args.local_steps, round_hook=coord, max_steps=K, host_loss_every_step=True)
        loop.global_step = 0
        barrier_sync(device)
        r0 = coord.round
        e0.record()
        loop.train(1)
        if coord.round == r0:
            coord.finish_round()
        e1.record()
        barrier_sync(device)
        ms_e2e = max_over_ranks(e0.elapsed_time(e1), device)
        result["e2e"] = {"value": tokens / ms_e2e * 1e3, "unit": "tokens/s", "ms_per_step": ms_e2e / K,
                         "h2d_bytes_per_step": host_data.bytes_per_batch, "d2h_bytes_per_step": 4,
                         "api": "training_manager.DeltaLoop.train",
                         "last_loss": float(loop.host_losses[(K - 1) % loop.host_losses.numel()]) if loop.host_losses is not None else None}
        coord.timer.summary()
    # ---- region 3: ONE WHOLE ROUND measured directly (BASELINE.json's second metric, avg-round wall time): local_steps
    # optimizer steps, delta emit, the reference-faithful learned mixer (meta_epochs^2 passes over val_texts sequences @ val_seq,
    # hivetrain/averaging_logic.py:490-541 + neurons/averager.py:106) executed by all ranks, averaging, base broadcast + reset ----
    if not args.no_full_round and learned and (world == 1 or ex is not None):
        coord.meta_epochs = args.meta_epochs
        nsteps_meta = args.meta_epochs ** 2 * len(val)
        barrier_sync(device)
        m0 = coord.meta_steps_done
        e0.record()
        for i in range(args.local_steps):
            trainer.step(dev_data.pool[i % len(dev_data.pool)])
        em = torch.cuda.Event(enable_timing=True)
        em.record()
        coord.finish_round()
        e1.record()
        # path (b): the step right after the round is launched WITHOUT any synchronisation in between -- its forward GEMMs acquire
        # the owners' base flags in-kernel while the pushed shards are still landing -- and compared with the step after it
        ef0, ef1, ef2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        ef0.record()
        trainer.step(dev_data.pool[0])
        ef1.record()
        trainer.step(dev_data.pool[1])
        ef2.record()
        barrier_sync(device)
        first_ms, next_ms = max_over_ranks(ef0.elapsed_time(ef1), device), max_over_ranks(ef1.elapsed_time(ef2), device)
        ms_round = max_over_ranks(e0.elapsed_time(e1), device)
        ms_mine = max_over_ranks(e0.elapsed_time(em), device)
        ph = coord.timer.summary()
        coord.meta_epochs = 0
        done = coord.meta_steps_done - m0

        result["full_round"] = {
            "measured_directly": True, "round_ms": round(ms_round, 2), "local_steps": args.local_steps,
            "mining_ms": round(ms_mine, 2), "exchange_ms": round(ms_round - ms_mine, 2), "meta_epochs": args.meta_epochs,
            "meta_steps": int(done), "meta_steps_expected": int(nsteps_meta),
            "ms_per_meta_step": round(max_over_ranks(ph.get("meta_learning", 0.0), device) / max(done, 1), 4),
            "phase_ms_rank0": {k: round(v, 3) for k, v in ph.items()},
            "val_set": {"texts": args.val_texts, "seq": Tv, "batch": Bv, "batches": len(val)},
            "tokens_per_s_incl_averaging": round(args.local_steps * B * T * world / ms_round * 1e3, 1),
            "first_step_after_round_ms": round(first_ms, 3), "ordinary_step_ms": round(next_ms, 3),
            "val_loss_last_step": float(coord.meta.loss_acc[1]) if coord.meta is not None else None,
            "w_mean_per_miner": [round(float(x), 5) for x in coord.w.mean(dim=1)]}
    # ---- cross-rank agreement: every rank must hold the same base after the rounds above ----
    cks = ops.checksum(trainer.base)
    if world > 1:
        allc = [None] * world
        dist.all_gather_object(allc, cks)
    else:
        allc = [cks]
    result["base_checksum"] = {"rank0": allc[0], "identical_on_all_ranks": bool(all(c == allc[0] for c in allc))}
    if hasattr(ex, "win"):
        ex.win.check_errors()
    if outputs is not None:
        write_outputs(args.dump_outputs, outputs)
    if dist.is_initialized():
        dist.destroy_process_group()
    return result if rank == 0 else {}


def main():
    args = parse_args()
    if args.dump_outputs and args.impl in ("reference", "torch-bf16"):
        raise SystemExit(f"--dump-outputs is not implemented for --impl {args.impl}")
    if args.impl == "reference":
        sys.path.insert(0, os.path.join(ROOT, "baseline"))
        from baseline.reference_arm import run_reference
        out = run_reference(args)
        if out:
            print(json.dumps(out), flush=True)
        return
    if args.impl == "torch-bf16":
        maybe_respawn(args)
        from baseline.torch_bf16_arm import run_torch_bf16
        out = run_torch_bf16(args)
        if out:
            print(json.dumps(out), flush=True)
        return
    maybe_respawn(args)
    out = run_ours(args)
    if out:
        print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
