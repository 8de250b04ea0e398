#!/usr/bin/env python
"""Headline benchmark: BERT-large pre-training throughput (sequences/s, whole job) on N B200s.

    python bench.py --gpus 1 --steps K --warmup W                 # this repo (fused sm_100a engine)
    python bench.py --impl reference --gpus 1 --steps K --warmup W  # unmodified reference + torch shims
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W    # N > 1, one rank per GPU over NCCL

Config = BASELINE.json phase 1 (`config/bert_pretraining_phase1_config.json`): BERT-large uncased
(L24 H1024 A16 I4096, vocab 30522 -> 30528), seq 128, micro-batch 96 per GPU, max 20 predictions,
masked_token_fraction 0.2, LAMB lr 6e-3 poly warm-up 0.2843, dropout 0.1, bf16 compute (the reference arm
runs its stock fp16 autocast + GradScaler).  ``--phase 2`` selects seq 512 / micro-batch 16 / 80 preds.
Synthetic data of that shape, random-init weights (no network for corpora/checkpoints).

One *step* = one optimizer step = ``--accum`` micro-batches (forward+backward each) + gradient
reduction over the ranks + LAMB update.  Default accumulation = the shipped 8-GPU arithmetic of the config
(`run_pretraining.py:218-228`: ceil(ceil(65536 / 8) / 96) = 86 micro-batches for phase 1, 256 for phase 2), i.e. on
8 GPUs the default run IS global batch 65536; fewer GPUs keep the per-GPU work (weak scaling).
``--global-batch G`` applies the shipped arithmetic to G for the actual world size.

After the headline config (phase 1, bf16) the same process measures BASELINE.json's other GPU configs for a few
steps each and reports them under ``extra.configs``: phase 2 (both arms), RoBERTa recipe with fp8 GEMM operands and
phase 1 + K-FAC (this repo only).  ``--no-extras`` skips them.  At N > 1 the fused reduce-scatter + LAMB + all-gather
kernel is first checked against NCCL all-reduce + single-GPU LAMB on the real arena (``extra.fused_parity_max_abs``)
and its in-kernel timeline is reported (``extra.fused_step_timeline``).

Timing: W >= 3 untimed warm-up steps, then exactly K steps bracketed by barrier + synchronize, CUDA
events on the launching stream, max over ranks; an L2 flush (256 MB write) precedes every step and the
per-step working set (~10 GB of activations) is far larger than the 126 MB L2 anyway; nvidia-smi
clocks/throttle reasons are sampled during the timed region.
``e2e`` repeats the measurement (at most 6 timed steps) through the public training API (`pretrain.forward_backward_pass` /
`take_optimizer_step`) with every micro-batch copied from pinned host memory inside the timed region and
the loss read back to the host every optimizer step.

``--dump-outputs DIR`` (this repository's arm, the config chosen on the command line) writes what the last timed step computed, after the
timing: ``DIR/loss.npy`` (float32, the loss of each micro-batch as ``forward_backward_pass`` returned it) and
``DIR/params_sample.npy`` (float32, the fp32 master weights after the LAMB update at DUMP_SAMPLE positions drawn
from a fixed seed).  Inputs, initial weights and dropout masks follow ``--seed``, so two builds run with the same
arguments can be compared output by output.  Compare with a tolerance: the gradient reductions are not bitwise
reproducible, and two runs of one build differed by up to 1.5e-5 in a micro-batch loss (~0.13) and 3e-6 in a sampled
weight (NVIDIA B200 at a 1000 W power limit, phase 1, 4 timed steps).
"""
from __future__ import annotations

import argparse
import json
import math
import os
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

PHASES = {
    1: dict(seq=128, local_batch=96, max_pred=20, lr=6e-3, warmup=0.2843, max_steps=7038, global_batch=65536),
    2: dict(seq=512, local_batch=16, max_pred=80, lr=4e-3, warmup=0.128, max_steps=1563, global_batch=32768),
}
# config #4 of BASELINE.json: RoBERTa-style recipe (config/roberta_pretraining_config.json + roberta_large_cased_config.json):
# no next-sentence task, cased 28996-token vocabulary, 15 % dynamic masking, linear decay
ROBERTA = dict(seq=512, local_batch=16, max_pred=80, lr=4e-4, warmup=0.06, max_steps=100000, global_batch=8192,
               vocab_size=28996, next_sentence=False, mask_prob=0.15, lr_decay="linear")
MODEL = dict(vocab_size=30522, hidden_size=1024, num_hidden_layers=24, num_attention_heads=16,
             intermediate_size=4096, max_position_embeddings=512, type_vocab_size=2)
DUMP_SAMPLE = 1 << 22            # weights kept by --dump-outputs: 16 MB of float32


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=4)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--phase", type=int, default=1, choices=[1, 2])
    ap.add_argument("--accum", type=int, default=0,
                    help="micro-batches per optimizer step (default: the shipped 8-GPU arithmetic of the config: 86 / 256 / 64)")
    ap.add_argument("--global-batch", type=int, default=0, help="use the shipped ceil arithmetic for this global batch")
    ap.add_argument("--local-batch", type=int, default=0)
    ap.add_argument("--backend", default="fused", choices=["nccl", "fused"],
                    help="gradient reduction (ours): fused = one peer-memory kernel for reduce-scatter + LAMB + all-gather")
    ap.add_argument("--layers", type=int, default=0, help="debug only: fewer layers (marks the result invalid)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="headline config only (skip extra.configs)")
    ap.add_argument("--fp8", action="store_true", help="fp8 GEMM operands (separate config; the headline stays bf16)")
    ap.add_argument("--roberta", action="store_true",
                    help="RoBERTa-style recipe (seq 512, no NSP, cased vocabulary, linear decay) instead of --phase; ours only")
    ap.add_argument("--kfac", action="store_true", help="K-FAC preconditioner on (BASELINE config #5); ours only")
    ap.add_argument("--seed", type=int, default=42)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's losses and a fixed sample of the updated weights as DIR/*.npy")
    return ap.parse_args()


def dist_setup(args):
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1 and not dist.is_initialized() and args.impl != "reference":   # the reference inits its own group
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", "29533")
        dist.init_process_group("nccl", init_method="env://", device_id=dev)
    return rank, world, local, dev


def synth_batches(n, B, S, vocab, max_pred, seed, dtype, pin=True, next_sentence=True, mask_prob=0.2):
    """n pre-masked micro-batches on the host: [ids, seg, mask, labels, nsp]."""
    import numpy as np
    import torch
    from bert_pytorch_b200.data import synthetic
    from bert_pytorch_b200.data.dataset import mask_batch, segment_ids_and_input_mask
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(n):
        ids, sp, nsl = synthetic.make_samples(B, S, vocab, next_sentence, rng)
        seg, im = segment_ids_and_input_mask(ids, sp)
        masked, labels = mask_batch(ids, sp, mask_token_index=4, max_pred_per_seq=max_pred, masked_lm_prob=mask_prob,
                                    vocab_size=vocab, rng=rng)
        ts = [torch.from_numpy(np.ascontiguousarray(a)).to(dtype) for a in (masked, seg, im, labels, nsl.astype(np.int32))]
        out.append([t.pin_memory() if pin else t for t in ts])
    return out


def timed_steps(run_step, K, W, flusher, dev):
    """W warm-up + K timed optimizer steps; returns (ms_per_step local, clocks record)."""
    import torch
    import torch.distributed as dist
    from bert_pytorch_b200.utils.timing import ClockSampler
    for i in range(W):
        flusher.flush()
        run_step(i)
    torch.cuda.synchronize()
    if dist.is_initialized():
        dist.barrier()
    torch.cuda.synchronize()
    sampler = ClockSampler(gpu_index=dev.index or 0)
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(K):
        flusher.flush()
        run_step(W + i)
    e1.record()
    torch.cuda.synchronize()
    if dist.is_initialized():
        dist.barrier()
    torch.cuda.synchronize()
    clocks = sampler.stop()
    return e0.elapsed_time(e1) / K, clocks


def dump_outputs(out_dir, losses, flat_param):
    """The last timed step's outputs as float32 .npy files (see the module docstring)."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    n = flat_param.numel()
    idx = np.sort(np.random.default_rng(1234).choice(n, min(n, DUMP_SAMPLE), replace=False))
    sample = flat_param[torch.from_numpy(idx).to(flat_param.device)]
    np.save(os.path.join(out_dir, "loss.npy"), torch.stack(losses).float().cpu().numpy())
    np.save(os.path.join(out_dir, "params_sample.npy"), sample.float().cpu().numpy())


def max_over_ranks(x, dev):
    import torch
    import torch.distributed as dist
    if not dist.is_initialized():
        return x
    t = torch.tensor([x], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def min_over_ranks(x, dev):
    return -max_over_ranks(-x, dev)


def fused_parity(comm, arena, opt, dev, rank, world):
    """Driver-side correctness proof of the fused reduce-scatter + LAMB + all-gather kernel (the driver's pytest box has
    one GPU): one optimizer step on the REAL arena with per-rank pseudo-random gradients, once as NCCL all-reduce(avg)
    + single-GPU arena LAMB and once through the peer-memory kernel; returns max |delta| over the bf16 weights every
    rank holds afterwards and the fp32 master shard it owns, max over ranks.  State is restored."""
    import torch
    import torch.distributed as dist
    from bert_pytorch_b200 import ops
    P0, M0, V0 = arena.flat_param.clone(), arena.exp_avg.clone(), arena.exp_avg_sq.clone()
    steps0 = [g.get("step", 0) for g in opt.param_groups]
    gen = torch.Generator(device=dev).manual_seed(4242 + rank)
    g = torch.randn(arena.numel, device=dev, generator=gen) * 0.05

    def restore():
        arena.flat_param.copy_(P0); arena.exp_avg.copy_(M0); arena.exp_avg_sq.copy_(V0)
        for grp, st in zip(opt.param_groups, steps0):
            grp["step"] = st
        arena.flat_grad.zero_()
    arena.flat_grad.copy_(g)
    dist.all_reduce(arena.flat_grad)
    arena.flat_grad.mul_(1.0 / world)
    ops.arena_lamb_step(arena, opt)
    ref = arena.flat_param.clone()
    restore()
    arena.flat_grad.copy_(g)
    torch.cuda.synchronize(); dist.barrier()
    comm.fused_lamb_step(opt, loss_scale=1.0)
    torch.cuda.synchronize()
    lo, hi = comm.lo, comm.hi
    d_master = (arena.flat_param[lo:hi] - ref[lo:hi]).abs().max().item() if hi > lo else 0.0
    d_shadow = (arena.flat_shadow.float() - ref.to(arena.flat_shadow.dtype).float()).abs().max().item()
    restore()
    arena.refresh_shadow()
    if hasattr(comm, "_master_stale"):
        comm._master_stale = False
    torch.cuda.synchronize(); dist.barrier()
    return {"fp32_master_shard": max_over_ranks(d_master, dev), "bf16_weights_all_ranks": max_over_ranks(d_shadow, dev)}


# ------------------------------------------------------------------------------------------------
# this repository
# ------------------------------------------------------------------------------------------------
def run_ours(args, ph, B, accum, rank, world, dev):
    import torch
    from bert_pytorch_b200 import BertConfig, ops, pretrain
    from bert_pytorch_b200.models import BertForPreTraining, BertPretrainingCriterion
    from bert_pytorch_b200.models.arena import NO_DECAY_KEYS, ParamArena
    from bert_pytorch_b200.ops import api as K
    from bert_pytorch_b200.optim import GradScaler, Lamb, LinearWarmUpScheduler, PolyWarmUpScheduler
    from bert_pytorch_b200.parallel import DataParallel, make_comm
    from bert_pytorch_b200.utils.timing import L2Flusher
    assert ops.available(), "sm_100a extension not loaded"
    torch.manual_seed(args.seed + rank)
    vocab = ph.get("vocab_size", MODEL["vocab_size"])
    cfg = BertConfig.from_dict(dict(MODEL, vocab_size=vocab, next_sentence=ph.get("next_sentence", True), hidden_act="gelu",
                                    hidden_dropout_prob=0.1, attention_probs_dropout_prob=0.1, initializer_range=0.02))
    if args.layers:
        cfg.num_hidden_layers = args.layers
    cfg.pad_vocab(8)
    cfg.max_predictions_per_seq = ph["max_pred"]
    model = BertForPreTraining(cfg).to(dev)
    arena = ParamArena(model, device=dev)
    comm = make_comm(args.backend if world > 1 else None)
    if getattr(comm, "fuses_optimizer", False):
        try:
            comm.adopt(arena)        # arenas -> NVLink symmetric memory; reduction + LAMB become one kernel
        except Exception as e:       # no P2P fabric / symmetric memory on this box: the NCCL backend still works
            if rank == 0:
                print(f"[bench] fused backend unavailable ({type(e).__name__}: {e}); falling back to nccl", file=sys.stderr)
            comm = make_comm("nccl")
    ddp = DataParallel(model, comm=comm, arena=arena)
    named = list(model.named_parameters())
    groups = [{"params": [p for n, p in named if not any(k in n for k in NO_DECAY_KEYS)], "weight_decay": 0.01},
              {"params": [p for n, p in named if any(k in n for k in NO_DECAY_KEYS)], "weight_decay": 0.0}]
    opt = Lamb(groups, lr=ph["lr"])
    arena.bind_optimizer(opt)
    scaler = GradScaler(enabled=False)
    precond = None
    if args.kfac:                      # the runtime's K-FAC set-up (pretrain.prepare_optimizers, reference defaults)
        from bert_pytorch_b200 import kfac
        precond = kfac.KFAC(model, lr=ph["lr"], factor_decay=0.95, damping=0.003, kl_clip=0.001, factor_update_freq=1,
                            inv_update_freq=10, skip_layers=["BertLMPredictionHead", "embedding"],
                            comm_method=kfac.CommMethod.HYBRID_OPT, grad_worker_fraction=0.5, inv_dtype=torch.float16,
                            accumulate_data=False, compute_factor_in_hook=True, distribute_layer_factors=False,
                            grad_scaler=scaler, comm=ddp.comm)
    pretrain.configure_fused_reduction(ddp, precond)
    Sched = LinearWarmUpScheduler if ph.get("lr_decay") == "linear" else PolyWarmUpScheduler
    scheds = [Sched(opt, warmup=ph["warmup"], total_steps=ph["max_steps"])]
    if precond is not None:
        scheds.append(Sched(precond, warmup=ph["warmup"], total_steps=ph["max_steps"]))
    crit = BertPretrainingCriterion(cfg.vocab_size)
    model.train()
    if args.fp8:
        model.bert.fused_engine().enable_fp8()
    flusher = L2Flusher(dev)

    pool = synth_batches(8, B, ph["seq"], vocab, ph["max_pred"], args.seed + 17 * rank, torch.int32,
                         next_sentence=ph.get("next_sentence", True), mask_prob=ph.get("mask_prob", 0.2))
    dev_pool = [[t.to(dev) for t in b] for b in pool]
    loss_acc = torch.zeros((), device=dev)

    opt_events = []
    step_losses = []                   # the micro-batch losses of the latest step (device tensors, no sync)

    def step_device(i):
        step_losses.clear()
        for m in range(accum):
            batch = dev_pool[(i * accum + m) % len(dev_pool)]
            loss = pretrain.forward_backward_pass(ddp, crit, scaler, batch, accum, sync_grads=(m == accum - 1),
                                                  compute_dtype=torch.bfloat16)
            loss_acc.add_(loss)
            step_losses.append(loss.detach())
        for sc in scheds:
            sc.step()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        pretrain.take_optimizer_step(opt, precond, ddp, scaler)
        e1.record()
        opt_events.append((e0, e1))

    host_losses = []

    def step_e2e(i):
        # the public training API, inputs from pinned host memory, loss read back each optimizer step
        window = torch.zeros((), device=dev)
        for m in range(accum):
            hb = pool[(i * accum + m) % len(pool)]
            batch = [t.to(dev, non_blocking=True) for t in hb]
            window += pretrain.forward_backward_pass(ddp, crit, scaler, batch, accum, sync_grads=(m == accum - 1),
                                                     compute_dtype=torch.bfloat16)
        for sc in scheds:
            sc.step()
        pretrain.take_optimizer_step(opt, precond, ddp, scaler)
        host_losses.append(float(window))

    parity = None
    if world > 1 and getattr(comm, "fuses_optimizer", False) and precond is None:
        parity = fused_parity(comm, arena, opt, dev, rank, world)     # before anything is timed
    l0 = K.KERNEL_LAUNCHES
    ms, clocks = timed_steps(step_device, args.steps, args.warmup, flusher, dev)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, step_losses, arena.flat_param)
    timeline = None
    if world > 1 and hasattr(comm, "timeline") and precond is None:
        torch.cuda.synchronize()
        tl = comm.timeline()                                          # last timed step, this rank
        timeline = {k: [min_over_ranks(v, dev), max_over_ranks(v, dev)] for k, v in tl.items()}
    launches = (K.KERNEL_LAUNCHES - l0) * args.steps // (args.steps + args.warmup)
    e2e = None
    if not args.no_e2e:
        ke = min(args.steps, 6)
        ms_e2e, _ = timed_steps(step_e2e, ke, max(1, min(args.warmup, 2)), flusher, dev)
        h2d = sum(t.numel() * t.element_size() for t in pool[0]) * accum
        e2e = dict(ms=ms_e2e, h2d=h2d, d2h=4, steps=ke)
    final_loss = float(loss_acc) / max(1, (args.steps + args.warmup))
    torch.cuda.synchronize()
    opt_ms = [a.elapsed_time(b) for a, b in opt_events[args.warmup:args.warmup + args.steps]]
    opt_mean = max_over_ranks(sum(opt_ms) / max(1, len(opt_ms)), dev) if opt_ms else None
    what = ("K-FAC preconditioner step + gradient all-reduce + LAMB kernels" if args.kfac else
            "fused reduce-scatter + LAMB + all-gather kernel, INCLUDING its wait for the slowest rank's backward "
            "(the kernel alone: tools/peer_check.py --big)" if getattr(comm, "fuses_optimizer", False) and world > 1
            else "LAMB kernels (all-reduce happens in the last micro-step)" if world > 1 else "LAMB kernels")
    extra = dict(loss_mean=final_loss, backend=getattr(comm, "name", "single"),
                 optimizer_step_ms=None if opt_mean is None else round(opt_mean, 3), optimizer_step_is=what)
    if parity is not None:
        extra["fused_parity_max_abs"] = parity
    if timeline is not None:
        extra["fused_step_timeline"] = dict(timeline, note="[min, max] over ranks of the in-kernel %globaltimer split of the "
                                            "last timed step; barrier_wait_ms = wait for the slowest rank's backward pass")
    del ddp, model, arena, opt, comm, dev_pool, pool
    return ms, clocks, launches, e2e, extra


# ------------------------------------------------------------------------------------------------
# reference arm: the unmodified reference code path on torch-native shims
# ------------------------------------------------------------------------------------------------
def run_reference(args, ph, B, accum, rank, world, dev):
    shims, ref = os.path.join(ROOT, "baseline", "shims"), os.path.join(ROOT, "baseline", "_ref")
    if not os.path.isdir(ref) or not os.path.exists(os.path.join(ref, "run_pretraining.py")):
        return None
    sys.path[:0] = [shims, ref]
    import torch
    import run_pretraining as R          # the reference's own module
    from bert_pytorch_b200.data import synthetic  # only to write vocab/model json (no compute path)
    from bert_pytorch_b200.utils.timing import L2Flusher
    work = tempfile.mkdtemp(prefix=f"refbench_r{rank}_")
    vocab = synthetic.write_vocab(os.path.join(work, "vocab.txt"), MODEL["vocab_size"])
    layers = args.layers or MODEL["num_hidden_layers"]
    model_json = synthetic.write_model_config(os.path.join(work, "model.json"), vocab, **dict(MODEL, num_hidden_layers=layers))
    ns = argparse.Namespace(
        config_file=None, input_dir=work, output_dir=os.path.join(work, "out"), model_config_file=model_json,
        masked_token_fraction=0.2, max_predictions_per_seq=ph["max_pred"], disable_progress_bar=True,
        num_steps_per_checkpoint=10 ** 9, skip_checkpoint=True, checkpoint_activations=False, log_prefix="ref",
        seed=args.seed, fp16=True, learning_rate=ph["lr"], lr_decay="poly", warmup_proportion=ph["warmup"],
        global_batch_size=B * accum * world, local_batch_size=B, max_steps=float(ph["max_steps"]), steps=1e9,
        previous_phase_end_step=0, kfac=False, kfac_inv_interval=10, kfac_factor_interval=1, kfac_stat_decay=0.95,
        kfac_damping=0.003, kfac_kl_clip=0.001, kfac_skip_layers=["BertLMPredictionHead", "embedding"],
        local_rank=int(os.environ.get("LOCAL_RANK", 0)))
    os.makedirs(ns.output_dir, exist_ok=True)
    # the reference creates its output tree on the main process only but every rank lists it (run_pretraining.py:246);
    # with per-rank scratch directories each rank makes its own
    os.makedirs(os.path.join(ns.output_dir, "pretrain_ckpts"), exist_ok=True)
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    os.environ.setdefault("MASTER_PORT", "29534")
    os.environ.setdefault("RANK", "0")
    os.environ.setdefault("WORLD_SIZE", "1")
    torch.manual_seed(args.seed + rank)
    import torch.distributed as dist
    real_init = dist.init_process_group
    if dist.is_initialized():
        # second config in this process (extra.configs): the reference's setup_training() calls init_process_group
        # unconditionally (run_pretraining.py:185); the group of the headline run is still alive, so that one call
        # becomes a no-op -- re-initialising under torchrun's agent store hung a 2-GPU box for 10 minutes
        dist.init_process_group = lambda *a, **k: None
    try:
        ns = R.setup_training(ns)                  # init_process_group('nccl'), batch arithmetic
    finally:
        dist.init_process_group = real_init
    assert ns.accumulation_steps == accum, (ns.accumulation_steps, accum)
    model, checkpoint, global_step, criterion, ns = R.prepare_model(ns)       # BertForPreTraining + DDP
    optimizer, preconditioner, lr_schedulers, scaler = R.prepare_optimizers(ns, model, checkpoint, global_step)
    model.train()
    flusher = L2Flusher(dev)
    pool = synth_batches(8, B, ph["seq"], MODEL["vocab_size"], ph["max_pred"], args.seed + 17 * rank, torch.int64)
    dev_pool = [[t.to(dev) for t in b] for b in pool]

    def one_step(i, batches_of, read_loss):
        avg = 0.0
        for m in range(accum):
            batch = batches_of((i * accum + m) % len(pool))
            loss = R.forward_backward_pass(model, criterion, scaler, batch, ns.accumulation_steps,
                                           sync_grads=(m == accum - 1))
            if read_loss:
                avg += loss.item()          # the reference loop syncs every micro-step (run_pretraining.py:542)
        for lrs in lr_schedulers:
            lrs.step()
        R.take_optimizer_step(optimizer, preconditioner, model, scaler)
        return avg

    step_device = lambda i: one_step(i, lambda j: dev_pool[j], False)
    step_e2e = lambda i: one_step(i, lambda j: [t.to(ns.device) for t in pool[j]], True)
    ms, clocks = timed_steps(step_device, args.steps, args.warmup, flusher, dev)
    e2e = None
    if not args.no_e2e:
        ke = min(args.steps, 6)
        ms_e2e, _ = timed_steps(step_e2e, ke, max(1, min(args.warmup, 2)), flusher, dev)
        h2d = sum(t.numel() * t.element_size() for t in pool[0]) * accum
        e2e = dict(ms=ms_e2e, h2d=h2d, d2h=4 * accum, steps=ke)
    extra = dict(backend="nccl-ddp", scaler=float(scaler.get_scale()))
    del model, optimizer, dev_pool, pool
    return ms, clocks, 0, e2e, extra


def roofline(args, ph, seq_per_s_per_gpu: float) -> dict:
    """Model FLOPs per sequence as executed (GEMMs + attention, forward + backward = 3x forward; the MLM head on the
    masked rows only for this repo, on every position for the reference) against the MEASURED sustained cuBLAS bf16
    throughput of this pool (MEASURED_PEAKS.json; the profiling recipe's fallback when the file is absent)."""
    try:
        H, I, L, S = 1024, 4096, args.layers or 24, ph["seq"]
        V = (ph.get("vocab_size", 30522) + 7) // 8 * 8
        head_rows = ph["max_pred"] if args.impl == "ours" else S
        fwd = S * L * (2 * (4 * H * H + 2 * H * I) + 4 * S * H) + head_rows * (2 * H * H + 2 * H * V)
        gflop = 3 * fwd / 1e9
        peak, src = 1590.0, "fallback"
        path = os.path.join(ROOT, "MEASURED_PEAKS.json")
        if os.path.exists(path):
            with open(path) as f:
                mp = json.load(f)
            peak = float(mp.get("bf16_tflops_sustained") or mp.get("bf16_tflops") or peak)
            src = "MEASURED_PEAKS.json bf16_tflops_sustained"
        tflops = seq_per_s_per_gpu * gflop / 1e3
        return {"gflop_per_seq": round(gflop, 1), "tflops_per_gpu": round(tflops, 1), "peak_tflops": peak,
                "peak_source": src, "fraction_of_peak": round(tflops / peak, 3)}
    except Exception as e:  # noqa: BLE001 - diagnostics only, never fail the benchmark line
        return {"error": repr(e)}


def shipped_accum(ph) -> int:
    """Micro-batches per optimizer step of the shipped config on 8 GPUs (run_pretraining.py:218-228 arithmetic)."""
    return math.ceil(math.ceil(ph["global_batch"] / 8) / ph["local_batch"])


def run_config(args, rank, world, dev):
    """One config on one arm -> the JSON record (rank 0 prints it)."""
    ph = dict(ROBERTA) if args.roberta else dict(PHASES[args.phase])
    B = args.local_batch or ph["local_batch"]
    if args.global_batch:
        accum = math.ceil(math.ceil(args.global_batch / world) / B)
    else:
        accum = args.accum or shipped_accum(ph)
    global_batch = B * accum * world
    fn = run_reference if args.impl == "reference" else run_ours
    res = fn(args, ph, B, accum, rank, world, dev)
    if res is None:
        return None
    ms_local, clocks, launches, e2e, extra = res
    ms = max_over_ranks(ms_local, dev)
    value = global_batch / (ms / 1e3)
    extra = dict(extra)
    extra["roofline"] = roofline(args, ph, value / world)
    ours = args.impl == "ours"
    out = {
        "metric": (f"RoBERTa-large recipe (seq{ph['seq']}, no NSP)" if args.roberta else f"BERT-large phase{args.phase} (seq{ph['seq']})")
        + (" + K-FAC" if args.kfac else "") + " pretraining sequences/sec, whole job, device-timed max over ranks",
        "value": round(value, 2), "unit": "sequences/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": round(ms, 3), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": ("fp8 GEMM operands (e4m3 fwd / e5m2 grads, per-tensor delayed scaling) + bf16" if args.fp8 else "bf16")
        if ours else "fp16 (reference stock AMP)", "data": "synthetic",
        "impl": args.impl,
        "config": {"model": ("roberta-large-cased (BERT-large, no NSP) L24 H1024 A16 I4096 V29000" if args.roberta
                             else "bert-large-uncased L24 H1024 A16 I4096 V30528")
                   + (f" [DEBUG layers={args.layers}]" if args.layers else ""), "kfac": bool(args.kfac),
                   "global_batch": global_batch, "seq_len": ph["seq"], "local_batch": B, "accumulation_steps": accum,
                   "shipped_global_batch": ph["global_batch"], "max_predictions_per_seq": ph["max_pred"],
                   "optimizer": "LAMB", "dropout": 0.1,
                   "dtype": "bf16 operands, fp32 accumulate / master" + (" + fp8 GEMM operands" if args.fp8 else "") if ours
                   else "fp16 autocast + GradScaler (stock)",
                   "mlm_head": "masked-only (max_predictions_per_seq rows per sequence, same loss)" if ours
                   else "dense (every position, as the reference computes it)",
                   "parallelism": f"dp{world}", "grad_reduction": extra.get("backend"),
                   "l2": "256MB L2 flush before every step; per-step working set (~10 GB activations) >> 126 MB L2",
                   "note": "step = one optimizer step of accumulation_steps micro-batches incl. gradient reduction + LAMB; "
                           "default accumulation = shipped global batch on 8 GPUs (per-GPU work fixed: weak scaling)"},
        "clocks": {"sm_mhz": clocks.get("sm_mhz"), "sm_max_mhz": clocks.get("sm_max_mhz"),
                   "reasons": clocks.get("reasons"), "power_w_max": clocks.get("power_w_max"),
                   "samples": clocks.get("samples")},
        "gpu_launches": int(launches),
        "extra": extra,
    }
    if e2e is not None:
        ms_e = max_over_ranks(e2e["ms"], dev)
        out["e2e"] = {"value": round(global_batch / (ms_e / 1e3), 2), "unit": "sequences/s",
                      "h2d_bytes_per_step": int(e2e["h2d"]), "d2h_bytes_per_step": int(e2e["d2h"]),
                      "ms_per_step": round(ms_e, 3), "steps": int(e2e.get("steps", args.steps))}
    return out


def compact(rec: dict) -> dict:
    """What extra.configs keeps of a sub-run."""
    if rec is None:
        return {"unavailable": "not measured"}
    keep = {k: rec[k] for k in ("metric", "value", "unit", "ms_per_step", "steps", "warmup", "dtype", "gpu_launches") if k in rec}
    keep["config"] = {k: rec["config"][k] for k in ("global_batch", "seq_len", "local_batch", "accumulation_steps", "kfac",
                                                     "mlm_head", "grad_reduction") if k in rec["config"]}
    keep["clocks"] = rec.get("clocks")
    ex = rec.get("extra", {})
    keep["extra"] = {k: ex[k] for k in ("loss_mean", "optimizer_step_ms", "roofline") if k in ex}
    return keep


def main():
    args = parse()
    if args.impl == "reference" and not os.path.exists(os.path.join(ROOT, "baseline", "_ref", "run_pretraining.py")):
        print(json.dumps({"impl": "reference", "unavailable": "baseline/_ref missing: the reference has no "
                          "setup.py/pyproject.toml so pip cannot install it; copy /root/reference there"}))
        return
    import torch
    if not torch.cuda.is_available():
        print(json.dumps({"impl": args.impl, "unavailable": "no CUDA device"}))
        return
    if args.dump_outputs and args.impl != "ours":
        sys.exit("--dump-outputs dumps this repository's timed path; it is not available with --impl reference")
    if (args.roberta or args.kfac) and args.impl != "ours":
        print(json.dumps({"impl": args.impl, "unavailable": "--roberta / --kfac are measured for this repository only "
                          "(the reference arm runs the two headline configs)"}))
        return
    rank, world, local, dev = dist_setup(args)
    assert world == max(1, args.gpus) or world == 1, f"WORLD_SIZE={world} but --gpus {args.gpus}"
    out = run_config(args, rank, world, dev)
    if out is None:
        if rank == 0:
            print(json.dumps({"impl": "reference", "unavailable": "reference copy not found under baseline/_ref"}))
        return
    headline = args.phase == 1 and not (args.roberta or args.kfac or args.fp8 or args.layers)
    # An extra config that fails on ONE rank leaves the others inside a collective: nothing after that point may
    # depend on the process group.  Ranks signal through a flag file (one node), a watcher thread on every rank ends the
    # process when it appears -- rank 0 prints the headline line (plus whatever extras finished) first.
    import threading
    state = {"out": out, "configs": None, "printed": False}
    flag = os.path.join("/tmp", f"b200_bench_abort_{os.environ.get('MASTER_PORT', '0')}_{os.getppid()}")
    lock = threading.Lock()

    def emit():
        with lock:
            if rank == 0 and not state["printed"]:
                if state["configs"] is not None:
                    state["out"]["extra"]["configs"] = state["configs"]
                print(json.dumps(state["out"]), flush=True)
                state["printed"] = True

    def watch():
        while not os.path.exists(flag):
            time.sleep(0.5)
        emit()
        os._exit(0)

    if world > 1:
        threading.Thread(target=watch, daemon=True).start()
    if headline and not args.no_extras:
        # BASELINE.json configs #3-#5 in the same process, a few steps each (reduced accumulation: more optimizer /
        # reduction share per unit compute than the shipped config, i.e. conservative)
        import gc
        subs = [("phase2", dict(phase=2, accum=16))]
        if args.impl == "ours":
            subs += [("roberta_fp8", dict(roberta=True, fp8=True, accum=16)), ("kfac", dict(kfac=True, accum=16))]
        configs = state["configs"] = {}
        for name, over in subs:
            sub = argparse.Namespace(**vars(args))
            sub.steps, sub.warmup, sub.no_e2e, sub.global_batch = min(args.steps, 4), 3, True, 0
            sub.dump_outputs = None
            for k, v in over.items():
                setattr(sub, k, v)
            gc.collect()
            torch.cuda.empty_cache()
            # an extra config that HANGS (a wedged collective) must not cost the headline line either: after `limit`
            # seconds the flag file goes up, every rank's watcher prints what there is (rank 0) and leaves
            limit = float(os.environ.get("B200_BENCH_EXTRA_TIMEOUT", "420"))

            def _expired(name=name):
                if state["configs"] is not None:
                    state["configs"].setdefault(name, {"error": f"timeout: no result after {limit:.0f} s"})
                try:
                    open(flag, "w").close()
                except OSError:
                    pass
                if world == 1:
                    emit()
                    os._exit(0)
            guard = threading.Timer(limit, _expired)
            guard.daemon = True
            guard.start()
            try:
                configs[name] = compact(run_config(sub, rank, world, dev))
                guard.cancel()
            except Exception as e:  # noqa: BLE001 - an extra config must never cost the headline line
                guard.cancel()
                configs[name] = {"error": f"{type(e).__name__}: {e}"[:300]}
                if world > 1:       # the other ranks may be blocked in a collective: stop here, everywhere
                    emit()
                    open(flag, "w").close()
                    time.sleep(2.0)
                    os._exit(0)
    emit() if rank == 0 else None
    if world > 1:                   # a wedged communicator must not turn a finished measurement into a timeout
        threading.Timer(30.0, lambda: os._exit(0)).start()
    import torch.distributed as dist
    if dist.is_initialized():
        dist.destroy_process_group()
    if world > 1:
        sys.stdout.flush()
        os._exit(0)


if __name__ == "__main__":
    main()
