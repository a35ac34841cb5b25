"""Run the UNMODIFIED reference GPTModel (baseline/_ref) on CPU/gloo and dump loss + grads (test helper, run as a script).

The reference assumes CUDA in three places that do not touch the math (device of the RoPE table, the default causal mask, the
CUDA RNG tracker around dropout with p=0).  This harness patches those call sites from the outside; no reference file is edited.

    torchrun/spawn env: RANK WORLD_SIZE MASTER_ADDR MASTER_PORT;  argv: out_prefix tp [grads | save <dir> | load <dir>]
"""
import contextlib
import json
import os
import sys
import zlib

import torch

REPO = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.join(REPO, "baseline", "_ref"))
sys.path = [p for p in sys.path if os.path.abspath(p or ".") != REPO]
torch.cuda.current_device = lambda: torch.device("cpu")
torch.cuda.synchronize = lambda *a, **k: None


class _HostStream:
    """Stand-in for the side streams the reference creates for device-to-host copies (MoE all-to-all dispatcher): on CPU everything is synchronous."""

    def __init__(self, *a, **k):
        pass

    def wait_stream(self, *a, **k):
        pass

    def synchronize(self):
        pass

    def record_event(self, *a, **k):
        return self

    def wait_event(self, *a, **k):
        pass

    wait = query = lambda self, *a, **k: True




def _cpu_device_factories():
    """The reference spells ``device='cuda'`` literally in a few factory calls (optimizer scale tensors, found-inf flags): send those to the CPU."""
    def wrap(fn):
        def inner(*a, **k):
            d = k.get("device")
            if d is not None and "cuda" in str(d):
                k["device"] = "cpu"
            return fn(*a, **k)
        return inner
    for name in ("tensor", "zeros", "ones", "empty", "full", "zeros_like", "ones_like", "empty_like", "arange", "randn", "rand"):
        setattr(torch, name, wrap(getattr(torch, name)))


_cpu_device_factories()
_orig_type = torch.Tensor.type


def _type(self, *a, **k):
    """``tensor.type()`` is compared against 'torch.cuda.FloatTensor' in the reference's gradient clipping: report CPU tensors under the CUDA name."""
    if not a and not k:
        r = _orig_type(self)
        return r if r.startswith("torch.cuda") else r.replace("torch.", "torch.cuda.", 1)
    return _orig_type(self, *a, **k)


torch.Tensor.type = _type
torch.Tensor.cuda = lambda self, *a, **k: self          # the reference's vision tower moves its position ids with .cuda()
torch.cuda.Stream = _HostStream
torch.cuda.Event = _HostStream
torch.cuda.current_stream = lambda *a, **k: _HostStream()
torch.cuda.stream = lambda *a, **k: contextlib.nullcontext()
import torch.distributed as dist  # noqa: E402


def seeded_full(name, shape, std=0.05):
    g = torch.Generator().manual_seed(zlib.crc32(name.encode()))
    return torch.empty(shape).normal_(0, std, generator=g)


def init_params(named_params, tp_rank, tp_world):
    """Same rule as bench.py::deterministic_init: FULL tensor from a name-seeded generator, then this rank's slice."""
    with torch.no_grad():
        for n, p in named_params:
            if p.dim() == 1:
                p.fill_(1.0)
                continue
            sharded = bool(getattr(p, "tensor_model_parallel", False)) and tp_world > 1
            dim = int(getattr(p, "partition_dim", -1))
            shape = list(p.shape)
            if sharded:
                shape[dim] *= tp_world
            full = seeded_full(n, shape)
            if sharded and n.endswith("linear_fc1.weight"):
                # SwiGLU: the logical matrix is [gate; up]; a TP rank holds [gate chunk r; up chunk r] (TP-size-invariant model)
                g, u = full.chunk(2, dim=0)
                p.copy_(torch.cat([g.chunk(tp_world, dim=0)[tp_rank], u.chunk(tp_world, dim=0)[tp_rank]], dim=0))
            else:
                p.copy_(full.chunk(tp_world, dim=dim)[tp_rank] if sharded else full)


CFG = dict(num_layers=2, hidden_size=64, ffn_hidden_size=128, num_attention_heads=4, num_query_groups=2, kv_channels=16, vocab=128, seq=32, batch=2)
CFG.update(json.loads(os.environ.get("REF_MODEL_SIZE", "{}")))          # the checkpoint-interop runs use a smaller model


# REF_VARIANT=moe: 4 experts, top-2, softmax-then-top-k router with the switch aux loss, all-gather dispatcher, one expert MLP per expert (no grouped GEMM)
_V = os.environ.get("REF_VARIANT", "")
MOE_KW = dict(num_moe_experts=4, moe_router_topk=2, moe_token_dispatcher_type="allgather", moe_router_load_balancing_type="aux_loss",
              moe_aux_loss_coeff=0.02, moe_grouped_gemm=False, moe_ffn_hidden_size=96, **({"expert_model_parallel_size": 2} if _V == "moe_ep2" else {})) if _V.startswith("moe") else {}
if _V == "moe_dsv3":        # DeepSeek-V3 style router: sigmoid scores, group-limited top-k, scaling factor, per-sequence aux loss, z-loss, one shared expert
    MOE_KW.update(num_moe_experts=8, moe_router_topk=4, moe_router_score_function="sigmoid", moe_router_num_groups=2, moe_router_group_topk=1, moe_router_topk_scaling_factor=2.5,
                  moe_router_load_balancing_type="seq_aux_loss", moe_aux_loss_coeff=0.01, moe_z_loss_coeff=1e-3, moe_shared_expert_intermediate_size=64, moe_ffn_hidden_size=48,
                  moe_router_pre_softmax=False)
if _V == "moe_drop":        # capacity-limited routing: drop by probability, pad every expert's input to the capacity; the all-to-all dispatcher (EP = 1: no communication)
    MOE_KW.update(moe_token_dispatcher_type="alltoall", moe_expert_capacity_factor=1.0, moe_token_drop_policy="probs", moe_pad_expert_input_to_capacity=True,
                  moe_router_pre_softmax=True)
if _V.startswith("moe"):
    import json as _json

    MOE_KW.update(_json.loads(os.environ.get("REF_MOE_OVERRIDE", "{}")))


def tokens():
    return torch.randint(0, CFG["vocab"], (CFG["batch"], CFG["seq"] + 1), generator=torch.Generator().manual_seed(1))


def main():
    out_prefix, tp = sys.argv[1], int(sys.argv[2])
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    dist.init_process_group("gloo", rank=rank, world_size=world)
    import torch.nn.functional as F
    import megatron.core.tensor_parallel as _tp
    import megatron.core.tensor_parallel.random as _tpr
    from megatron.core import parallel_state
    from megatron.core.models.gpt.gpt_layer_specs import get_gpt_layer_local_spec
    from megatron.core.models.gpt.gpt_model import GPTModel
    from megatron.core.transformer.transformer_config import TransformerConfig

    class _NoRng:
        def fork(self, *a, **k):
            return contextlib.nullcontext()

    _tp.get_cuda_rng_tracker = _tpr.get_cuda_rng_tracker = lambda *a, **k: _NoRng()
    if _V == "pp2":
        return pp_main(out_prefix, rank, F, TransformerConfig, GPTModel, get_gpt_layer_local_spec, parallel_state)
    parallel_state.initialize_model_parallel(tensor_model_parallel_size=tp, **({"expert_model_parallel_size": 2} if _V == "moe_ep2" else {}))
    if _V == "bert":
        return bert_main(out_prefix, rank, F, TransformerConfig)
    if _V == "t5":
        return t5_main(out_prefix, rank, TransformerConfig)
    if _V == "vit":
        return vit_main(out_prefix, rank, TransformerConfig)
    cfg = TransformerConfig(
        num_layers=CFG["num_layers"], hidden_size=CFG["hidden_size"], ffn_hidden_size=CFG["ffn_hidden_size"], num_attention_heads=CFG["num_attention_heads"],
        num_query_groups=CFG["num_query_groups"], kv_channels=CFG["kv_channels"], normalization="RMSNorm", gated_linear_unit=True, activation_func=F.silu,
        add_bias_linear=False, hidden_dropout=0.0, attention_dropout=0.0, use_cpu_initialization=True, bias_activation_fusion=False, bias_dropout_fusion=False,
        masked_softmax_fusion=False, gradient_accumulation_fusion=False, perform_initialization=False, tensor_model_parallel_size=tp,
        **MOE_KW, **json.loads(os.environ.get("REF_CFG_OVERRIDE", "{}")),
    )
    spec = get_gpt_layer_local_spec(num_experts=MOE_KW.get("num_moe_experts"), moe_grouped_gemm=False, normalization="RMSNorm") if MOE_KW else get_gpt_layer_local_spec(normalization="RMSNorm")
    m = GPTModel(cfg, spec, vocab_size=CFG["vocab"], max_sequence_length=CFG["seq"], parallel_output=True,
                 share_embeddings_and_output_weights=False, position_embedding_type="rope", rotary_base=10000)
    mode = sys.argv[3] if len(sys.argv) > 3 else "grads"
    if mode in ("save", "load"):
        # checkpoint interop: the reference writes (or reads back) a torch_dist distributed checkpoint of this model
        from megatron.core import dist_checkpointing

        ckpt_dir = sys.argv[4]
        tp_rank = parallel_state.get_tensor_model_parallel_rank()
        if mode == "save":
            init_params(m.named_parameters(), tp_rank, tp)
            dist_checkpointing.save(m.sharded_state_dict(), ckpt_dir)
        else:
            with torch.no_grad():
                for _, p in m.named_parameters():
                    p.zero_()
            sd = dist_checkpointing.load(m.sharded_state_dict(), ckpt_dir)
            m.load_state_dict(sd, strict=False)
            got = {n: p.detach().clone() for n, p in m.named_parameters()}
            init_params(m.named_parameters(), tp_rank, tp)       # what the writer initialised
            worst = max(float((got[n] - p.detach()).abs().max()) for n, p in m.named_parameters())
            torch.save({"max_abs_diff": worst, "n_params": len(got)}, f"{out_prefix}.rank{rank}.pt")
        dist.barrier()
        dist.destroy_process_group()
        return
    init_params(m.named_parameters(), parallel_state.get_tensor_model_parallel_rank(), tp)
    tok = tokens()
    if _V == "moe_ep2":                      # EP ranks are data-parallel ranks for the dense part: each sees its own half of the batch
        tok = tok[rank:rank + 1]
    s = CFG["seq"]
    pos = torch.arange(s).unsqueeze(0).expand(tok.shape[0], -1).contiguous()
    mask = torch.triu(torch.ones(s, s), diagonal=1).bool()[None, None]
    if _V in ("optim", "distopt"):
        dist_opt = _V == "distopt"
        if dist_opt:                       # DP = 2: every rank trains on its own sample
            tok = tok[rank:rank + 1]
            pos = pos[:1]
        # three optimizer steps through the reference's optimizer stack (param groups with / without weight decay, global-norm clipping, the LR scheduler)
        from megatron.core.optimizer import OptimizerConfig, get_megatron_optimizer
        from megatron.core.optimizer_param_scheduler import OptimizerParamScheduler

        ocfg = OptimizerConfig(optimizer="adam", lr=1e-2, min_lr=1e-3, weight_decay=0.1, adam_beta1=0.9, adam_beta2=0.95, adam_eps=1e-8, clip_grad=0.5, bf16=False, fp16=False,
                               use_distributed_optimizer=dist_opt)
        from megatron.core.distributed import DistributedDataParallel, DistributedDataParallelConfig

        m = DistributedDataParallel(cfg, DistributedDataParallelConfig(grad_reduce_in_fp32=True, overlap_grad_reduce=False, use_distributed_optimizer=dist_opt), m)
        opt = get_megatron_optimizer(ocfg, [m])
        sched = OptimizerParamScheduler(opt, init_lr=0.0, max_lr=1e-2, min_lr=1e-3, lr_warmup_steps=2, lr_decay_steps=10, lr_decay_style="cosine", start_wd=0.1, end_wd=0.1,
                                        wd_incr_steps=10, wd_incr_style="constant")
        losses, norms = [], []
        for it in range(3):
            m.zero_grad_buffer()
            opt.zero_grad()
            loss = m(tok[:, :-1].contiguous(), pos, mask, labels=tok[:, 1:].contiguous()).float().mean()
            loss.backward()
            m.finish_grad_sync()
            ok, gn, _ = opt.step()
            sched.step(increment=1)
            losses.append(float(loss))
            norms.append(float(gn))
        torch.save({"losses": losses, "grad_norms": norms, "lr": [g["lr"] for g in opt.param_groups], "params": {n: p.detach().clone() for n, p in m.module.named_parameters()}},
                   f"{out_prefix}.rank{rank}.pt")
        dist.barrier()
        dist.destroy_process_group()
        return
    loss = m(tok[:, :-1].contiguous(), pos, mask, labels=tok[:, 1:].contiguous()).float().mean()
    loss.backward()
    torch.save({"loss": float(loss), "grads": {n: p.grad.clone() for n, p in m.named_parameters()}}, f"{out_prefix}.rank{rank}.pt")
    dist.barrier()
    dist.destroy_process_group()


def bert_main(out_prefix, rank, F, TransformerConfig):
    """BERT (learned positions, token types, LM head + binary head, padding mask) from the reference's local spec."""
    from megatron.core.models.bert.bert_layer_specs import bert_layer_local_spec
    from megatron.core.models.bert.bert_model import BertModel

    cfg = TransformerConfig(num_layers=2, hidden_size=64, ffn_hidden_size=128, num_attention_heads=4, hidden_dropout=0.0, attention_dropout=0.0, use_cpu_initialization=True,
                            bias_activation_fusion=False, bias_dropout_fusion=False, masked_softmax_fusion=False, gradient_accumulation_fusion=False, perform_initialization=False,
                            layernorm_epsilon=1e-5)
    m = BertModel(cfg, num_tokentypes=2, transformer_layer_spec=bert_layer_local_spec, vocab_size=128, max_sequence_length=32, parallel_output=True, add_binary_head=True)
    init_params(m.named_parameters(), 0, 1)
    with torch.no_grad():
        for n, p in m.named_parameters():
            if p.dim() == 1 and ("bias" in n):
                p.copy_(seeded_full(n, list(p.shape), 0.02))
    g = torch.Generator().manual_seed(3)
    tok = torch.randint(0, 128, (2, 32), generator=g)
    types = torch.randint(0, 2, (2, 32), generator=g)
    pad = torch.ones(2, 32, dtype=torch.long)
    pad[1, 25:] = 0
    labels = torch.randint(0, 128, (2, 32), generator=g)
    lm_loss, binary = m(tok, pad, tokentype_ids=types, lm_labels=labels)
    loss = (lm_loss.float() * pad).sum() / pad.sum() + binary.float().logsumexp(-1).mean()
    loss.backward()
    torch.save({"loss": float(loss), "grads": {n: p.grad.clone() for n, p in m.named_parameters() if p.grad is not None}}, f"{out_prefix}.rank{rank}.pt")
    dist.barrier()
    dist.destroy_process_group()


def t5_inputs():
    g = torch.Generator().manual_seed(5)
    b, se, sd = 2, 24, 12
    enc = torch.randint(0, 128, (b, se), generator=g)
    dec = torch.randint(0, 128, (b, sd), generator=g)
    labels = torch.randint(0, 128, (b, sd), generator=g)
    enc_keep = torch.ones(b, se)
    enc_keep[1, 20:] = 0
    enc_mask = enc_keep[:, :, None] * enc_keep[:, None, :]                                  # [b, se, se] 1 = attend
    dec_mask = torch.tril(torch.ones(sd, sd))[None].expand(b, -1, -1).contiguous()
    x_mask = torch.ones(b, sd, 1) * enc_keep[:, None, :]
    return enc, dec, enc_mask, dec_mask, x_mask, labels


def t5_main(out_prefix, rank, TransformerConfig):
    """T5 encoder-decoder (learned positions, cross attention, shared embeddings + LM head bias) from the reference's local block specs."""
    from megatron.core.models.T5.t5_model import T5Model
    from megatron.core.models.T5.t5_spec import get_t5_decoder_with_local_block_spec, get_t5_encoder_with_local_block_spec

    kw = dict(hidden_size=64, ffn_hidden_size=128, num_attention_heads=4, kv_channels=16, hidden_dropout=0.0, attention_dropout=0.0, use_cpu_initialization=True,
              bias_activation_fusion=False, bias_dropout_fusion=False, masked_softmax_fusion=False, gradient_accumulation_fusion=False, perform_initialization=False)
    cfg, enc_cfg = TransformerConfig(num_layers=2, **kw), TransformerConfig(num_layers=2, **kw)
    m = T5Model(cfg, enc_cfg, get_t5_encoder_with_local_block_spec(2), get_t5_decoder_with_local_block_spec(2), vocab_size=128, max_sequence_length=32, parallel_output=True,
                share_embeddings_and_output_weights=True)
    init_params(m.named_parameters(), 0, 1)
    with torch.no_grad():
        for n, p in m.named_parameters():
            if p.dim() == 1 and "bias" in n:
                p.copy_(seeded_full(n, list(p.shape), 0.02))
    enc, dec, enc_mask, dec_mask, x_mask, labels = t5_inputs()
    loss = m(enc, dec, (enc_mask < 0.5).unsqueeze(1), (dec_mask < 0.5).unsqueeze(1), (x_mask < 0.5).unsqueeze(1), lm_labels=labels).float().mean()
    loss.backward()
    torch.save({"loss": float(loss), "grads": {n: p.grad.clone() for n, p in m.named_parameters() if p.grad is not None}}, f"{out_prefix}.rank{rank}.pt")
    dist.barrier()
    dist.destroy_process_group()


def pp_main(out_prefix, rank, F, TransformerConfig, GPTModel, get_gpt_layer_local_spec, parallel_state):
    """Pipeline parallel 2 (1F1B, 4 micro-batches) through the reference's schedule: 4 layers, 2 per stage, untied embeddings."""
    from functools import partial

    from megatron.core.pipeline_parallel import get_forward_backward_func

    # (the interleaved schedule of the reference does not produce self-consistent losses over gloo — its batched p2p exchanges same-shaped tensors in both
    # directions without tags — so only the non-interleaved schedule is compared; our interleaved schedule is checked against the single-process model elsewhere)
    parallel_state.initialize_model_parallel(pipeline_model_parallel_size=2)
    pre, post = parallel_state.is_pipeline_first_stage(), parallel_state.is_pipeline_last_stage()
    cfg = TransformerConfig(num_layers=4, hidden_size=64, ffn_hidden_size=128, num_attention_heads=4, num_query_groups=2, kv_channels=16, normalization="RMSNorm",
                            gated_linear_unit=True, activation_func=F.silu, add_bias_linear=False, hidden_dropout=0.0, attention_dropout=0.0, use_cpu_initialization=True,
                            bias_activation_fusion=False, bias_dropout_fusion=False, masked_softmax_fusion=False, gradient_accumulation_fusion=False, perform_initialization=False,
                            pipeline_model_parallel_size=2, pipeline_dtype=torch.float32)
    m = GPTModel(cfg, get_gpt_layer_local_spec(normalization="RMSNorm"), vocab_size=128, max_sequence_length=32, pre_process=pre, post_process=post, parallel_output=True,
                 share_embeddings_and_output_weights=False, position_embedding_type="rope", rotary_base=10000)
    # layer names are LOCAL (layers.0 / layers.1 on both stages): seed by the GLOBAL name so that stage 1 holds layers 2 and 3 of the same 4-layer model
    off = 0 if pre else 2
    with torch.no_grad():
        for n, p in m.named_parameters():
            gname = n
            if ".layers." in n:
                head, rest = n.split(".layers.")
                i, tail = rest.split(".", 1)
                gname = f"{head}.layers.{int(i) + off}.{tail}"
            p.fill_(1.0) if p.dim() == 1 else p.copy_(seeded_full(gname, list(p.shape)))
    toks = torch.randint(0, 128, (4, 2, 33), generator=torch.Generator().manual_seed(2))            # 4 micro-batches of 2 sequences
    mask = torch.triu(torch.ones(32, 32), diagonal=1).bool()[None, None]
    pos = torch.arange(32).unsqueeze(0).expand(2, -1).contiguous()

    def loss_func(output):
        loss = output.float().mean()
        return loss, {"lm loss": loss.detach().clone()}

    def forward_step(data_iterator, model):
        t = next(data_iterator)
        return model(t[:, :-1].contiguous(), pos, mask, labels=t[:, 1:].contiguous()), loss_func

    fb = get_forward_backward_func()
    out = fb(forward_step_func=forward_step, data_iterator=iter(toks), model=[m], num_microbatches=4, seq_length=32, micro_batch_size=2, forward_only=False)
    losses = [float(d["lm loss"]) for d in out] if post else []
    torch.save({"losses": losses, "grads": {n: p.grad.clone() for n, p in m.named_parameters() if p.grad is not None}}, f"{out_prefix}.rank{rank}.pt")
    dist.barrier()
    dist.destroy_process_group()


def vit_main(out_prefix, rank, TransformerConfig):
    """CLIP ViT tower (conv patch embedding, class token, learned positions, pre-norm, bidirectional attention) from the reference's local layer spec."""
    from megatron.core.models.vision.clip_vit_model import CLIPViTModel
    from megatron.core.models.vision.vit_layer_specs import get_vit_layer_with_local_spec
    from megatron.core.transformer.torch_norm import WrappedTorchNorm

    cfg = TransformerConfig(num_layers=2, hidden_size=64, ffn_hidden_size=128, num_attention_heads=4, hidden_dropout=0.0, attention_dropout=0.0, use_cpu_initialization=True,
                            bias_activation_fusion=False, bias_dropout_fusion=False, masked_softmax_fusion=False, gradient_accumulation_fusion=False, perform_initialization=False)
    m = CLIPViTModel(cfg, get_vit_layer_with_local_spec(), ln_pre_impl=WrappedTorchNorm, ln_post_impl=WrappedTorchNorm, patch_dim=14, img_h=28, img_w=28)
    init_params(m.named_parameters(), 0, 1)
    with torch.no_grad():
        for n, p in m.named_parameters():
            if p.dim() == 1 and "bias" in n:
                p.copy_(seeded_full(n, list(p.shape), 0.02))
            if p.dim() > 2:
                p.copy_(seeded_full(n, list(p.shape), 0.05))
    x = torch.randn(2, 3, 28, 28, generator=torch.Generator().manual_seed(7))
    out = m(x)
    w = torch.randn(out.shape, generator=torch.Generator().manual_seed(8))
    loss = (out.float() * w).mean()
    loss.backward()
    torch.save({"loss": float(loss), "shape": tuple(out.shape), "grads": {n: p.grad.clone() for n, p in m.named_parameters() if p.grad is not None}}, f"{out_prefix}.rank{rank}.pt")
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
