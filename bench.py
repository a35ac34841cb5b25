#!/usr/bin/env python
"""Headline benchmark: Llama-3-8B training throughput at TP=N, bf16 compute, fp32 main grads.

    python bench.py --gpus 1 --steps 5 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus 8 --steps 5 --warmup 3
    python bench.py --impl reference ...      # unmodified NVIDIA/Megatron-LM from baseline/_ref
    python bench.py --gpus 1 --steps 5 --warmup 3 --dump-outputs OUT   # + OUT/*.npy: loss and weight sample after the last timed step

Both arms print ONE JSON line on rank 0 with the IDENTICAL ``metric`` string and the same workload:

  * the same Llama-3-8B architecture, TP=N **without** sequence parallelism (the stock reference's local norm
    asserts ``not sequence_parallel``), ``selective(core_attn)`` activation recompute, fp32 main-grad accumulation
    (reference default with ``--bf16``: ``megatron/training/arguments.py:1204-1217``), AdamW(lr 1e-5, wd 0.1,
    betas 0.9/0.95, clip 1.0), global batch 4 x seq 8192, micro-batch 1;
  * the same initial weights (every parameter generated from a name-seeded generator as the FULL tensor and
    sliced to this TP rank's shard) and the same synthetic tokens, so ``loss_by_step`` of the two arms is
    comparable step by step (tolerance: bf16 noise);
  * ``value`` = whole-job tokens/s, device-timed with CUDA events around exactly K optimizer steps, max over ranks.

The repo arm additionally reports the configuration it is designed for (TP=N + sequence parallel through the fused
AG->GEMM / GEMM->RS kernels, no recompute) under ``config.sp_variant`` — NOT comparable with the reference arm
(which cannot run SP), reported for the scaling picture only.
"""
from __future__ import annotations

import argparse
import gc
import json
import math
import os
import subprocess
import sys
import tempfile
import time
import zlib

REPO = os.path.dirname(os.path.abspath(__file__))
os.environ.setdefault("PYTORCH_CUDA_ALLOC_CONF", "expandable_segments:True")

METRIC = "tokens/sec (whole job, device-timed, max over ranks), Llama-3-8B TP=N, bf16 compute, fp32 main grads, no sequence parallel, selective(core_attn) recompute"
LLAMA3_8B = dict(num_layers=32, hidden=4096, ffn=14336, heads=32, groups=8, kv=128, vocab=128256, seq=8192)
# a warm-up-sized learning rate: with lr 3e-4 from step 1 (no warm-up) the first Adam steps move every weight by 1.5 % and the loss curve is
# chaotic (12.6 -> 4.3 -> 9.4 ...), so round-off differences between the arms would be amplified instead of compared
LR, MIN_LR, WD, CLIP, BETA1, BETA2 = 1e-5, 1e-6, 0.1, 1.0, 0.9, 0.95
DATA_SEED = 17


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=4)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--model", default="llama3_8b")
    ap.add_argument("--global-batch", type=int, default=4, help="sequences per optimizer step")
    ap.add_argument("--micro-batch", type=int, default=1)
    ap.add_argument("--seq", type=int, default=None)
    ap.add_argument("--layers", type=int, default=None, help="DEV ONLY: fewer layers (result is flagged invalid)")
    ap.add_argument("--tp-comm", default=None, choices=[None, "nccl", "nvlink", "fused"])
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-sp-variant", action="store_true", help="skip the second (TP=N + sequence parallel) measurement of the repo arm")
    ap.add_argument("--recompute", default="auto")
    ap.add_argument("--main-grads", default="fp32", choices=["fp32", "bf16"])
    ap.add_argument("--dtype", default="bf16", choices=["bf16", "mxfp8"], help="repo arm: mxfp8 = block-scaled E4M3 operands (tcgen05 kind::mxf8f6f4.block_scale) for every "
                    "linear layer's fprop/dgrad/wgrad GEMM (reference: --fp8-format e4m3 --fp8-recipe mxfp8), bf16 activations, fp32 master weights")
    # the other BASELINE.json configurations (repo arm): --model gpt3_6.7b | mixtral_8x7b | llama3_70b with their parallel layout
    ap.add_argument("--tp", type=int, default=None)
    ap.add_argument("--pp", type=int, default=None)
    ap.add_argument("--vp", type=int, default=None)
    ap.add_argument("--ep", type=int, default=None)
    ap.add_argument("--dispatcher", default=None, help="MoE token dispatcher: alltoall | allgather | flex (NVLink push/pull)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="repo arm: after the timed steps, write what the last timed step computed (its loss, every timed step's loss and a fixed, seeded sample of "
                         "the updated weights) to DIR/<name>.npy, so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs is implemented for --impl b200")
    return args


# BASELINE.json configs 3-5: (tp, pp, vp, ep) for 8 GPUs, global batch, recompute, main-grad dtype, sequence parallel
OTHER_CONFIGS = {
    "gpt3_6.7b": dict(tp=4, pp=2, vp=2, ep=1, global_batch=8, recompute={}, main_grads="fp32", sp=True,
                      metric="tokens/sec (whole job, device-timed, max over ranks), GPT-3 6.7B TP=4 x PP=2 interleaved 1F1B, bf16"),
    "mixtral_8x7b": dict(tp=1, pp=1, vp=None, ep=8, global_batch=8, recompute=dict(recompute_granularity="selective", recompute_modules=["core_attn"]), main_grads="fp32", sp=False,
                         metric="tokens/sec (whole job, device-timed, max over ranks), Mixtral 8x7B EP=8, bf16"),
    "llama3_70b": dict(tp=8, pp=1, vp=None, ep=1, global_batch=4, recompute=dict(recompute_granularity="full", recompute_method="uniform", recompute_num_layers=1), main_grads="bf16", sp=True,
                       metric="tokens/sec (whole job, device-timed, max over ranks), Llama-3 70B TP=8 + sequence parallel, distributed optimizer, bf16"),
}


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled every 200 ms during the timed region."""

    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index: int):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        self.idx = gpu_index

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200", "-i", str(self.idx)],
                                      stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.p is None:
            return out
        time.sleep(0.25)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [ln.strip().split(", ") for ln in open(self.f.name) if ln.strip()]
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            try:
                sm.append(float(r[1])), mx.append(float(r[2]))
                for n, v in zip(names, r[5:9]):
                    if v.strip().lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        if sm:
            sm.sort()
            out.update(sm_mhz=sm[len(sm) // 2], sm_max_mhz=max(mx), reasons=sorted(reasons), samples=len(sm))
        try:
            os.unlink(self.f.name)
        except OSError:
            pass
        return out


def env_rank():
    return int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("LOCAL_RANK", "0"))


def timed_loop(torch, dist, step_fn, steps, world):
    """barrier + sync, K steps between CUDA events, sync + barrier; returns max-over-ranks (device ms, wall ms)."""
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    for _ in range(steps):
        step_fn()
    e1.record()
    torch.cuda.synchronize()
    wall = (time.perf_counter() - t0) * 1e3
    if world > 1:
        dist.barrier()
    ms = torch.tensor([e0.elapsed_time(e1), wall], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    return float(ms[0]), float(ms[1])


def synthetic_tokens(torch, n_seq, seq, vocab, n_steps):
    """The benchmark's data: a DIFFERENT batch of uniform random token ids for every optimizer step, [n_steps, n_seq, seq+1]
    (inputs = [..., :-1], labels = [..., 1:]); the same stream in both arms (seeded CPU generator)."""
    g = torch.Generator().manual_seed(DATA_SEED)
    return torch.randint(0, vocab, (n_steps, n_seq, seq + 1), generator=g, dtype=torch.int64)


def deterministic_init(torch, named_params, tp_rank, tp_world, num_layers):
    """Identical initial weights for both arms and every TP size: each parameter is generated as the FULL
    (unsharded) fp32 tensor on the device from a generator seeded by crc32(name), then this rank's slice along
    ``partition_dim`` is copied into the local shard.  Matrices ~ N(0, 0.02) (output projections scaled by
    1/sqrt(2L) like Megatron's ``scaled_init_method_normal``), norm weights = 1, biases = 0."""
    gen = torch.Generator(device="cuda")
    n = 0
    with torch.no_grad():
        for name, p in named_params:
            name = name.replace("module.", "")
            if p.dim() == 1:
                p.fill_(1.0 if "norm" in name and name.endswith("weight") else 0.0)
                continue
            sharded = bool(getattr(p, "tensor_model_parallel", False)) and tp_world > 1
            dim = int(getattr(p, "partition_dim", -1))
            full_shape = list(p.shape)
            if sharded:
                full_shape[dim] *= tp_world
            gen.manual_seed(zlib.crc32(name.encode()))
            std = 0.02 / math.sqrt(2.0 * num_layers) if (".linear_proj." in name or ".linear_fc2." in name) else 0.02
            full = torch.empty(full_shape, dtype=torch.float32, device="cuda").normal_(0.0, std, generator=gen)
            if sharded and name.endswith("linear_fc1.weight"):
                # SwiGLU: the logical matrix is [gate; up]; a TP rank holds [gate chunk r; up chunk r] — the model is then the SAME function at every TP size
                ga, up = full.chunk(2, dim=0)
                shard = torch.cat([ga.chunk(tp_world, dim=0)[tp_rank], up.chunk(tp_world, dim=0)[tp_rank]], dim=0)
            else:
                shard = full.chunk(tp_world, dim=dim)[tp_rank] if sharded else full
            p.copy_(shard.to(p.dtype))
            del full
            n += 1
    return n


DUMP_SAMPLES_PER_PARAM = 4096      # 291 Llama-3-8B tensors -> 1.2 M fp32 values, 4.5 MiB: far below the 64 MiB the dump may take


def dump_outputs(torch, out_dir, model_chunks, timed_losses):
    """What the timed path computed in its last step, as float32 ``.npy`` files: ``loss.npy`` (that step's mean loss), ``loss_by_step.npy`` (one value
    per timed step) and ``param_sample.npy`` — this rank's updated weights, for each parameter (in ``named_parameters`` order) the elements at
    ``DUMP_SAMPLES_PER_PARAM`` flat indices drawn by a CPU generator seeded with crc32(name), so the same positions are sampled in every run."""
    import numpy as np

    os.makedirs(out_dir, exist_ok=True)
    losses = torch.stack([l.detach().float().reshape(()) for l in timed_losses]).cpu().numpy()
    samples = []
    with torch.no_grad():
        for chunk in model_chunks:
            for name, p in chunk.named_parameters():
                name = name.replace("module.", "")
                flat = p.detach().reshape(-1)
                g = torch.Generator().manual_seed(zlib.crc32(name.encode()))
                idx = torch.randint(0, flat.numel(), (min(flat.numel(), DUMP_SAMPLES_PER_PARAM),), generator=g)
                samples.append(flat[idx.to(flat.device)].float().cpu())
    np.save(os.path.join(out_dir, "loss.npy"), losses[-1:].astype(np.float32))
    np.save(os.path.join(out_dir, "loss_by_step.npy"), losses.astype(np.float32))
    np.save(os.path.join(out_dir, "param_sample.npy"), torch.cat(samples).numpy().astype(np.float32))


def losses_to_dict(torch, loss_tensors):
    vals = torch.stack([l.detach().float().reshape(()) for l in loss_tensors]).cpu().tolist() if loss_tensors else []
    return {str(i + 1): round(float(v), 5) for i, v in enumerate(vals)}


# ------------------------------------------------------------------------------------------------
def _b200_variant(args, torch, dist, rank, world, local, *, sequence_parallel, recompute, main_grads_fp32, want_e2e, sample_clocks, dump_dir=None):
    """Build a TrainEngine, run W warm-up + K timed steps (+ the e2e loop).  Returns a dict of plain floats.  With ``dump_dir``, rank 0 writes the
    outputs of the last timed step there before the e2e loop changes the weights."""
    from megatron_b200 import ops
    from megatron_b200.training.engine import TrainEngine

    overrides = {}
    if args.layers:
        overrides["num_layers"] = args.layers
    if args.dtype == "mxfp8":
        overrides.update(fp8="e4m3", fp8_recipe="mxfp8")
    eng = TrainEngine(args.model, tensor_model_parallel_size=world, sequence_parallel=sequence_parallel, micro_batch_size=args.micro_batch,
                      global_batch_size=args.global_batch, seq_length=args.seq, bf16=True, model_overrides=overrides, lr=LR, min_lr=MIN_LR,
                      weight_decay=WD, clip_grad=CLIP, grad_reduce_in_fp32=main_grads_fp32, **recompute)
    from megatron_b200.core import parallel_state as ps

    n_init = 0
    for chunk in eng.model_chunks:
        n_init += deterministic_init(torch, chunk.named_parameters(), ps.get_tensor_model_parallel_rank(), world, eng.preset["num_layers"])
    eng.optimizer.reload_model_params()
    n_total = args.warmup + 2 * args.steps + 1
    host = synthetic_tokens(torch, eng.num_microbatches * args.micro_batch, eng.seq_length, eng.preset["vocab_size"], n_total).pin_memory()
    dev_tokens = host.to("cuda")
    losses = []

    def step_dev():
        losses.append(eng.train_step(dev_tokens[len(losses)]))

    def step_e2e():
        losses.append(eng.train_step(host[len(losses)]))     # H2D copy of this step's tokens from pinned memory
        return float(losses[-1])                             # D2H read of the step's loss every step

    for _ in range(args.warmup):
        step_dev()
    sampler = ClockSampler(local)
    if rank == 0 and sample_clocks:
        sampler.start()
    ops.reset_launch_count()
    ms, _wall = timed_loop(torch, dist, step_dev, args.steps, world)
    launches = ops.launch_count()
    clocks = sampler.stop() if (rank == 0 and sample_clocks) else {}
    if dump_dir and rank == 0:
        dump_outputs(torch, dump_dir, eng.model_chunks, losses[args.warmup:])
    tokens_per_step = args.global_batch * eng.seq_length
    res = {"value": tokens_per_step * args.steps / (ms / 1e3), "ms_per_step": ms / args.steps, "gpu_launches": launches, "clocks": clocks,
           "tflops_per_gpu": eng.flops_per_step * args.steps / (ms / 1e3) / world / 1e12, "seq_length": eng.seq_length, "params_initialised": n_init}
    if want_e2e:
        step_e2e()
        _, e_wall = timed_loop(torch, dist, step_e2e, args.steps, world)
        res["e2e"] = {"value": tokens_per_step * args.steps / (e_wall / 1e3), "unit": "tokens/s", "h2d_bytes_per_step": host[0].numel() * host.element_size(),
                      "d2h_bytes_per_step": 4, "timing": "host wall clock incl. H2D of the step's tokens from pinned memory and D2H loss read, max over ranks"}
    res["loss_by_step"] = losses_to_dict(torch, losses)
    res["peak_mem_gib"] = torch.cuda.max_memory_allocated() / 2**30
    # drop every reference to the engine so a second variant fits
    del eng, dev_tokens, losses, step_dev, step_e2e
    gc.collect()
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats()
    return res


def run_b200_other(args):
    """Repo arm for the other BASELINE.json configurations (PP / EP / 70B).  Same timing contract; synthetic data; the model's own random init."""
    import torch
    import torch.distributed as dist

    sys.path.insert(0, REPO)
    rank, world, local = env_rank()
    assert world == args.gpus, f"launched with WORLD_SIZE={world} but --gpus {args.gpus}"
    from megatron_b200 import ops
    from megatron_b200.core import parallel_state as ps
    from megatron_b200.training import engine as _engine

    torch.cuda.set_device(local)
    _engine.initialize_distributed()
    c = dict(OTHER_CONFIGS.get(args.model, dict(tp=1, pp=1, vp=None, ep=1, global_batch=world, recompute={}, main_grads="fp32", sp=False, metric=f"tokens/sec, {args.model}")))
    tp, pp, vp, ep = args.tp or c["tp"], args.pp or c["pp"], args.vp if args.vp is not None else c["vp"], args.ep or c["ep"]
    if world < tp * pp:          # fewer GPUs than the named layout: shrink TP first (DEV runs)
        tp = max(1, world // pp)
    if pp == 1:
        vp = None
    dp = world // (tp * pp)
    ep = min(ep, dp * tp) if ep > 1 else 1
    gb = args.global_batch if args.global_batch != 4 or args.model not in OTHER_CONFIGS else c["global_batch"]
    gb = max(gb, dp * args.micro_batch * (pp if pp > 1 else 1))
    overrides = {}
    if args.layers:
        overrides["num_layers"] = args.layers
    if args.dispatcher:
        overrides["moe_token_dispatcher_type"] = args.dispatcher
    fp32_grads = (args.main_grads if args.main_grads != "fp32" or args.model not in OTHER_CONFIGS else c["main_grads"]) == "fp32"
    eng = _engine.TrainEngine(args.model, tensor_model_parallel_size=tp, pipeline_model_parallel_size=pp, virtual_pipeline_model_parallel_size=vp,
                              expert_model_parallel_size=ep, sequence_parallel=c["sp"] and tp > 1, micro_batch_size=args.micro_batch, global_batch_size=gb,
                              seq_length=args.seq, bf16=True, model_overrides=overrides, lr=LR, min_lr=MIN_LR, weight_decay=WD, clip_grad=CLIP,
                              grad_reduce_in_fp32=fp32_grads, **c["recompute"])
    n_total = args.warmup + 2 * args.steps + 1
    per_rank = eng.num_microbatches * args.micro_batch
    g = torch.Generator().manual_seed(DATA_SEED + ps.get_data_parallel_rank())
    host = torch.randint(0, eng.preset["vocab_size"], (n_total, per_rank, eng.seq_length + 1), generator=g, dtype=torch.int64).pin_memory()
    dev_tokens = host.to("cuda")
    losses = []

    def step_dev():
        losses.append(eng.train_step(dev_tokens[len(losses)]))

    def step_e2e():
        losses.append(eng.train_step(host[len(losses)]))
        return float(losses[-1])

    for _ in range(args.warmup):
        step_dev()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ops.reset_launch_count()
    ms, _ = timed_loop(torch, dist, step_dev, args.steps, world)
    launches = ops.launch_count()
    clocks = sampler.stop() if rank == 0 else {}
    if args.dump_outputs:
        # the loss lives on the last pipeline stage: rank 0 writes the max over ranks of each timed step's value (other stages report 0)
        timed = torch.stack([l.detach().float().reshape(()) for l in losses[args.warmup:]]).cuda()
        dist.all_reduce(timed, op=dist.ReduceOp.MAX)
        if rank == 0:
            dump_outputs(torch, args.dump_outputs, eng.model_chunks, list(timed))
    tokens_per_step = gb * eng.seq_length
    value = tokens_per_step * args.steps / (ms / 1e3)
    e2e = None
    if not args.no_e2e:
        step_e2e()
        _, e_wall = timed_loop(torch, dist, step_e2e, args.steps, world)
        e2e = {"value": tokens_per_step * args.steps / (e_wall / 1e3), "unit": "tokens/s", "h2d_bytes_per_step": host[0].numel() * 8, "d2h_bytes_per_step": 4}
    # the loss lives on the last pipeline stage: take the max over ranks of the per-step values (other stages report 0)
    lv = torch.stack([l.detach().float().reshape(()) for l in losses]).cuda()
    dist.all_reduce(lv, op=dist.ReduceOp.MAX)
    peak = torch.tensor([torch.cuda.max_memory_allocated() / 2**30], device="cuda")
    dist.all_reduce(peak, op=dist.ReduceOp.MAX)
    if rank == 0:
        print(json.dumps({
            "metric": c["metric"], "value": value, "unit": "tokens/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "bf16", "data": "synthetic (fresh random token batch per step; random-init weights)",
            "impl": "b200", "tflops_per_gpu": eng.flops_per_step * args.steps / (ms / 1e3) / world / 1e12, "loss_by_step": {str(i + 1): round(float(v), 5) for i, v in enumerate(lv.tolist())},
            "peak_mem_gib_max_over_ranks": float(peak), "gpu_launches": launches, "clocks": clocks, "e2e": e2e,
            "config": {"model": args.model + (f"[layers={args.layers} DEV-INVALID]" if args.layers else ""), "global_batch": gb, "micro_batch": args.micro_batch,
                       "seq_len": eng.seq_length, "parallelism": f"tp{tp}" + ("+sp" if c["sp"] and tp > 1 else "") + f" pp{pp}" + (f" vp{vp}" if vp else "") + f" ep{ep} dp{dp}",
                       "num_microbatches": eng.num_microbatches, "main_grads": "fp32" if fp32_grads else "bf16", "recompute": c["recompute"] or "none",
                       "moe_dispatcher": getattr(eng.config, "moe_token_dispatcher_type", None) if eng.config.num_moe_experts else None,
                       "l2_policy": "inputs larger than L2 (weights + activations stream through the 126 MB L2 every step)"},
        }), flush=True)
    try:
        dist.barrier()
        dist.destroy_process_group()
    except Exception:
        pass


def run_b200(args):
    import torch
    import torch.distributed as dist

    if args.model != "llama3_8b":
        return run_b200_other(args)
    sys.path.insert(0, REPO)
    rank, world, local = env_rank()
    assert world == args.gpus, f"launched with WORLD_SIZE={world} but --gpus {args.gpus}"
    if args.tp_comm:
        os.environ["MEGATRON_B200_TP_COMM"] = args.tp_comm
    from megatron_b200 import ops
    from megatron_b200.training import engine as _engine

    torch.cuda.set_device(local)
    _engine.initialize_distributed()
    fp32_grads = args.main_grads == "fp32"
    if args.recompute == "auto":
        # one GPU holds all 8B parameters + fp32 grads + optimizer state (135 GiB): also recompute the cheap ops' outputs
        mods = ["core_attn", "layernorm", "mlp_act"] if world == 1 else ["core_attn"]
        recompute = dict(recompute_granularity="selective", recompute_modules=mods)
    elif args.recompute == "full":
        recompute = dict(recompute_granularity="full", recompute_method="uniform", recompute_num_layers=1)
    elif args.recompute == "none":
        recompute = {}
    else:
        recompute = dict(recompute_granularity="selective", recompute_modules=args.recompute.split(","))

    main = _b200_variant(args, torch, dist, rank, world, local, sequence_parallel=False, recompute=recompute, main_grads_fp32=fp32_grads,
                         want_e2e=not args.no_e2e, sample_clocks=True, dump_dir=args.dump_outputs)
    # fused-vs-NCCL self check of every GEMM<->collective pair op on this model's shapes (N >= 2)
    pair_err = None
    if world > 1:
        try:
            from megatron_b200.parallel.selfcheck import pair_op_self_check

            pair_err = pair_op_self_check(dist.group.WORLD, seq=main["seq_length"], quick=True)
        except Exception as e:  # never lose the headline over the self check
            pair_err = {"error": f"{type(e).__name__}: {e}"[:200]}
    from megatron_b200.ops import gemm as _gemm
    from megatron_b200.parallel import fused as _fusedmod

    tp_mode = _fusedmod.get_mode(world_size=world) if world > 1 else "n/a"
    gemm_wins = {}
    for _key, _winner, _times in _gemm.tuning_report():
        gemm_wins[str(_winner).split(":")[0]] = gemm_wins.get(str(_winner).split(":")[0], 0) + 1
    attn_impl = ops.attention_impl_for(main["seq_length"], args.micro_batch, 32 // world) if hasattr(ops, "attention_impl_for") else "library"

    sp = None
    if world > 1 and not args.no_sp_variant:
        try:
            v = _b200_variant(args, torch, dist, rank, world, local, sequence_parallel=True, recompute={}, main_grads_fp32=fp32_grads,
                              want_e2e=False, sample_clocks=False)
            sp = {"parallelism": f"tp{world}+sp", "recompute": "none", "value": v["value"], "unit": "tokens/s", "ms_per_step": v["ms_per_step"],
                  "tflops_per_gpu": v["tflops_per_gpu"], "gpu_launches": v["gpu_launches"], "peak_mem_gib": v["peak_mem_gib"],
                  "loss_by_step": v["loss_by_step"], "note": "the design point of this repo (fused AG->GEMM / GEMM->RS kernels); the stock reference cannot run it"}
        except BaseException as e:  # noqa: BLE001 — the headline above must still be printed
            sp = {"error": f"{type(e).__name__}: {e}"[:300]}
    if rank == 0:
        mp = {}
        try:
            mp = json.load(open(os.path.join(REPO, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak_tf = mp.get("bf16_tflops_sustained", 1400.0)
        out = {
            "metric": METRIC + ("" if args.dtype == "bf16" else f" [{args.dtype} linear layers]"), "value": main["value"], "unit": "tokens/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": main["ms_per_step"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": args.dtype,
            "data": "synthetic (a fresh batch of uniform random token ids of the named shape every step, seed 17; name-seeded random-init weights identical in both arms)",
            "impl": "b200", "tflops_per_gpu": main["tflops_per_gpu"], "mfu_of_measured_sustained_cublas": main["tflops_per_gpu"] / peak_tf,
            "loss_by_step": main["loss_by_step"], "peak_mem_gib": main["peak_mem_gib"], "gpu_launches": main["gpu_launches"], "clocks": main["clocks"],
            "e2e": main.get("e2e"), "pair_op_max_rel_err": pair_err,
            "config": {"model": args.model + (f"[layers={args.layers} DEV-INVALID]" if args.layers else ""), "global_batch": args.global_batch,
                       "micro_batch": args.micro_batch, "seq_len": main["seq_length"], "parallelism": f"tp{world}", "sequence_parallel": False,
                       "l2_policy": "inputs larger than L2 (16 GB of bf16 weights + activations stream through the 126 MB L2 every step)",
                       "main_grads": args.main_grads, "optimizer": f"AdamW lr={LR} wd={WD} betas=({BETA1},{BETA2}) clip={CLIP}; fused multi-tensor kernel, fp32 master+moments",
                       "recompute": recompute or "none", "tp_comm": os.environ.get("MEGATRON_B200_TP_COMM", "auto"), "tp_comm_resolved": tp_mode,
                       "gemm": os.environ.get("MEGATRON_B200_GEMM", "auto"), "plain_gemm_shapes_tuned": gemm_wins, "attention": attn_impl,
                       "sp_variant": sp},
        }
        print(json.dumps(out), flush=True)
    try:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
    except Exception:
        pass


# ------------------------------------------------------------------------------------------------
def run_reference(args):
    """The UNMODIFIED reference (baseline/_ref, megatron-core 0.20.0) through its public API:
    parallel_state -> GPTModel(local spec) -> DistributedDataParallel -> get_megatron_optimizer ->
    get_forward_backward_func -> finalize_model_grads.  TransformerEngine/Apex are not installed, so
    this is the reference's stock "local" path (cuBLAS + NCCL, unfused attention, torch AdamW).
    Same workload as the repo arm (see the module docstring): TP=N without sequence parallelism,
    selective(core_attn) recompute, fp32 main grads, identical initial weights and tokens."""
    ref = os.path.join(REPO, "baseline", "_ref")
    if not os.path.isdir(os.path.join(ref, "megatron", "core")):
        print(json.dumps({"impl": "reference", "unavailable": "baseline/_ref is not installed (pip install --no-deps --target baseline/_ref <Megatron-LM checkout>)"}))
        return
    sys.path.insert(0, ref)
    sys.path = [p for p in sys.path if os.path.abspath(p or ".") != REPO]
    import warnings

    warnings.filterwarnings("ignore")
    import torch
    import torch.distributed as dist

    rank, world, local = env_rank()
    torch.cuda.set_device(local)
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    os.environ.setdefault("MASTER_PORT", "29512")
    os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "1")
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", local))
    try:
        import torch.nn.functional as F
        from megatron.core import parallel_state
        from megatron.core.distributed import DistributedDataParallel, DistributedDataParallelConfig
        from megatron.core.distributed.finalize_model_grads import finalize_model_grads
        from megatron.core.models.gpt.gpt_layer_specs import get_gpt_layer_local_spec
        from megatron.core.models.gpt.gpt_model import GPTModel
        from megatron.core.optimizer import OptimizerConfig, get_megatron_optimizer
        from megatron.core.pipeline_parallel.schedules import get_forward_backward_func
        from megatron.core.tensor_parallel.random import model_parallel_cuda_manual_seed
        from megatron.core.transformer.transformer_config import TransformerConfig
    except Exception as e:  # pragma: no cover
        if rank == 0:
            print(json.dumps({"impl": "reference", "unavailable": f"import failed: {type(e).__name__}: {e}"[:300]}))
        return

    P = dict(LLAMA3_8B)
    P["num_layers"] = args.layers or P["num_layers"]
    P["seq"] = args.seq or P["seq"]
    if args.model != "llama3_8b":
        if rank == 0:
            print(json.dumps({"impl": "reference", "unavailable": f"the reference arm drives the headline config (llama3_8b, TP=N) only; --model {args.model} is a repo-arm measurement"}))
        return
    parallel_state.initialize_model_parallel(tensor_model_parallel_size=world)
    model_parallel_cuda_manual_seed(1234)
    fp32_grads = args.main_grads == "fp32"

    def build(recompute):
        cfg = TransformerConfig(
            num_layers=P["num_layers"], hidden_size=P["hidden"], ffn_hidden_size=P["ffn"], num_attention_heads=P["heads"], num_query_groups=P["groups"],
            kv_channels=P["kv"], normalization="RMSNorm", gated_linear_unit=True, activation_func=F.silu, add_bias_linear=False, hidden_dropout=0.0,
            attention_dropout=0.0, tensor_model_parallel_size=world, sequence_parallel=False, bf16=True, params_dtype=torch.bfloat16,
            bias_activation_fusion=True, bias_dropout_fusion=True, masked_softmax_fusion=True, gradient_accumulation_fusion=False, **recompute,
        )
        m = GPTModel(cfg, get_gpt_layer_local_spec(normalization="RMSNorm"), vocab_size=P["vocab"], max_sequence_length=P["seq"], parallel_output=True,
                     share_embeddings_and_output_weights=False, position_embedding_type="rope", rotary_base=500000).cuda()
        n_init = deterministic_init(torch, m.named_parameters(), parallel_state.get_tensor_model_parallel_rank(), world, P["num_layers"])
        ddp = DistributedDataParallel(cfg, DistributedDataParallelConfig(grad_reduce_in_fp32=fp32_grads, overlap_grad_reduce=False, use_distributed_optimizer=True), m)
        opt = get_megatron_optimizer(OptimizerConfig(optimizer="adam", lr=LR, min_lr=MIN_LR, weight_decay=WD, bf16=True, params_dtype=torch.bfloat16,
                                                     clip_grad=CLIP, use_distributed_optimizer=True, adam_beta1=BETA1, adam_beta2=BETA2), [ddp])
        cfg.finalize_model_grads_func = finalize_model_grads
        cfg.no_sync_func = ddp.no_sync
        return cfg, ddp, opt, n_init

    nmb = args.global_batch // args.micro_batch
    n_total = args.warmup + 2 * args.steps + 1
    host = synthetic_tokens(torch, nmb * args.micro_batch, P["seq"], P["vocab"], n_total).pin_memory()
    dev_tokens = host.cuda()
    pos = torch.arange(P["seq"], device="cuda").unsqueeze(0).expand(args.micro_batch, -1).contiguous()
    fwd_bwd = get_forward_backward_func()

    def loss_func(out):
        loss = out.float().mean()
        # clone: the reference schedule scales the returned loss IN PLACE by 1/num_microbatches (schedules.py:343-346), which would
        # also rescale a detached alias of it
        return loss, {"lm loss": loss.detach().clone()}

    def fstep(it, model):
        b = next(it)
        return model(b[:, :-1].contiguous(), pos, None, labels=b[:, 1:].contiguous()), loss_func

    state = {}
    losses = []

    def make_step(tokens_fn, sync_loss):
        def step():
            t = tokens_fn()
            state["ddp"].zero_grad_buffer()
            state["opt"].zero_grad()
            it = iter(t[i * args.micro_batch : (i + 1) * args.micro_batch] for i in range(nmb))
            out = fwd_bwd(forward_step_func=fstep, data_iterator=it, model=state["ddp"], num_microbatches=nmb, seq_length=P["seq"],
                          micro_batch_size=args.micro_batch, forward_only=False)
            state["opt"].step()
            l = torch.stack([d["lm loss"] for d in out]).mean()
            losses.append(l)
            if sync_loss:
                return float(l)
        return step

    full = dict(recompute_granularity="full", recompute_method="uniform", recompute_num_layers=1)
    attempts = [("selective(core_attn)", dict(recompute_granularity="selective", recompute_modules=["core_attn"])),
                ("full(uniform,1)", full),
                ("full(uniform,1)+bf16-softmax", dict(full, attention_softmax_in_fp32=False))]
    if world == 1:
        # measured on the 180 GB part: selective recompute OOMs at TP=1 (fp32 [32,8192,8192] scores on top of
        # >= 120 GiB of parameter/optimizer state) and a failed attempt fragments the heap — start from full recompute
        attempts = attempts[1:]
    if os.environ.get("REF_RECOMPUTE"):
        attempts = [a for a in attempts if a[0].startswith(os.environ["REF_RECOMPUTE"])] or attempts
    used = None
    n_init = 0
    for name, rc in attempts:
        try:
            state.clear()
            losses.clear()
            torch.cuda.empty_cache()
            state["cfg"], state["ddp"], state["opt"], n_init = build(rc)
            step_dev = make_step(lambda: dev_tokens[len(losses)], False)
            for _ in range(args.warmup):
                step_dev()
            torch.cuda.synchronize()
            used = name
            break
        except torch.cuda.OutOfMemoryError as e:
            if rank == 0:
                print(f"[reference] OOM with recompute={name}: {str(e)[:300]}", file=sys.stderr, flush=True)
            state.clear()
            gc.collect()
            torch.cuda.empty_cache()
            continue
    ok = torch.tensor([1 if used else 0], device="cuda")
    if world > 1:
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
    if not int(ok):
        if rank == 0:
            print(json.dumps({"impl": "reference", "metric": METRIC, "n_gpus": world,
                              "unavailable": "reference local path runs out of memory on this config even with full activation recompute (unfused fp32 [32,8192,8192] attention scores + torch AdamW temporaries on top of the parameter/optimizer state)"}))
        return
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ms, _ = timed_loop(torch, dist, step_dev, args.steps, world)
    clocks = sampler.stop() if rank == 0 else {}
    tokens_per_step = args.global_batch * P["seq"]
    value = tokens_per_step * args.steps / (ms / 1e3)
    e2e = None
    if not args.no_e2e:
        step_e2e = make_step(lambda: host[len(losses)].cuda(non_blocking=True), True)
        step_e2e()
        _, e_wall = timed_loop(torch, dist, step_e2e, args.steps, world)
        e2e = {"value": tokens_per_step * args.steps / (e_wall / 1e3), "unit": "tokens/s", "h2d_bytes_per_step": host[0].numel() * 8, "d2h_bytes_per_step": 4,
               "timing": "host wall clock incl. H2D of the step's tokens from pinned memory and D2H loss read, max over ranks"}
    loss_by_step = losses_to_dict(torch, losses)
    if rank == 0:
        print(json.dumps({
            "impl": "reference", "metric": METRIC, "value": value, "unit": "tokens/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "bf16",
            "data": "synthetic (a fresh batch of uniform random token ids of the named shape every step, seed 17; name-seeded random-init weights identical in both arms)",
            "loss_by_step": loss_by_step, "clocks": clocks, "e2e": e2e, "peak_mem_gib": torch.cuda.max_memory_allocated() / 2**30,
            "config": {"model": args.model + (f"[layers={args.layers} DEV-INVALID]" if args.layers else ""), "global_batch": args.global_batch,
                       "micro_batch": args.micro_batch, "seq_len": P["seq"], "parallelism": f"tp{world}", "sequence_parallel": False,
                       "main_grads": args.main_grads, "optimizer": f"AdamW lr={LR} wd={WD} betas=({BETA1},{BETA2}) clip={CLIP}; torch.optim.AdamW behind megatron DistributedOptimizer",
                       "recompute": used, "params_initialised": n_init,
                       "backend": "megatron-core 0.20.0 local spec (TE/Apex absent): cuBLAS + NCCL + torch AdamW, unfused attention"},
        }), flush=True)
    if world > 1:
        dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_b200(a)
