"""Loss and gradient parity with the UNMODIFIED reference (megatron-core 0.20.0) on identical weights and tokens.

The same name-seeded full-tensor initialisation that ``bench.py`` applies to both arms is applied to a tiny Llama-style GPT in both
frameworks (TP=1 and TP=2 over gloo); forward loss and every parameter gradient must agree to fp32 round-off.  This is the contract
behind ``bench.py``'s ``loss_by_step`` comparison: same parameter names, same shard layout (interleaved QKV groups, [gate; up] fc1
halves), same math.

What the reference computed is stored under ``tests/golden/reference/`` (``tests/helpers/make_reference_golden.py`` regenerates it from an
install of the reference): losses, learning rates and norms in full; per tensor its shape, max |x|, sum, L2 norm and the values at a fixed
sample of elements; the reference's own checkpoints of the interop model; dataset samples; schedule tables."""
import json
import os
import sys

import pytest
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(REPO, "tests", "golden", "reference")


def _reference(name):
    """Per-rank results of the reference run ``name``."""
    with open(os.path.join(GOLDEN, f"model_{name}.json")) as f:
        return json.load(f)


def _assert_tensors_match(got, want, tol, what, relative=True):
    """Every tensor of ``want`` against this framework's full tensor in ``got``.  Each check follows from max |got - ref| < tol * scale, with
    scale = max |ref| (``relative``) or 1."""
    for n, w in want.items():
        g = got[n].detach().double()
        assert list(g.shape) == w["shape"], (what, n, list(g.shape), w["shape"])
        scale = max(w["absmax"], 1e-12) if relative else 1.0
        bound = tol * scale
        err = float((g.flatten()[w["idx"]] - torch.tensor(w["val"], dtype=torch.float64)).abs().max()) / scale
        assert err < tol, f"{what} {n}: err {err}"
        assert abs(float(g.abs().max()) - w["absmax"]) < bound, f"{what} {n}: max |x| {float(g.abs().max())} vs {w['absmax']}"
        assert abs(float(g.sum()) - w["sum"]) < bound * g.numel(), f"{what} {n}: sum {float(g.sum())} vs {w['sum']}"
        assert abs(float(g.norm()) - w["norm"]) < bound * g.numel() ** 0.5, f"{what} {n}: norm {float(g.norm())} vs {w['norm']}"


def _ours(rank, world, tp, variant=""):
    sys.path.insert(0, os.path.join(REPO, "tests", "helpers"))
    import torch.nn.functional as F

    from megatron_b200.core import parallel_state as ps
    from megatron_b200.core.models.gpt.gpt_layer_specs import get_gpt_layer_local_spec
    from megatron_b200.core.models.gpt.gpt_model import GPTModel
    from megatron_b200.core.transformer.transformer_config import TransformerConfig
    import zlib

    CFG = dict(num_layers=2, hidden_size=64, ffn_hidden_size=128, num_attention_heads=4, num_query_groups=2, kv_channels=16, vocab=128, seq=32, batch=2)
    ep2 = variant == "moe_ep2"
    ps.initialize_model_parallel(tensor_model_parallel_size=tp, **({"expert_model_parallel_size": 2} if ep2 else {}))
    cfg = TransformerConfig(
        num_layers=CFG["num_layers"], hidden_size=CFG["hidden_size"], ffn_hidden_size=CFG["ffn_hidden_size"], num_attention_heads=CFG["num_attention_heads"],
        num_query_groups=CFG["num_query_groups"], kv_channels=CFG["kv_channels"], normalization="RMSNorm", gated_linear_unit=True, activation_func=F.silu,
        add_bias_linear=False, hidden_dropout=0.0, attention_dropout=0.0, use_cpu_initialization=True, gradient_accumulation_fusion=False,
        perform_initialization=False, tensor_model_parallel_size=tp, **__import__("json").loads(os.environ.get("REF_CFG_OVERRIDE", "{}")),
        **(dict(num_moe_experts=4, moe_router_topk=2, moe_token_dispatcher_type="allgather", moe_router_load_balancing_type="aux_loss",
                moe_aux_loss_coeff=0.02, moe_grouped_gemm=False, moe_ffn_hidden_size=96, **({"expert_model_parallel_size": 2} if ep2 else {})) if variant.startswith("moe") else {}),
    )
    if variant == "moe_dsv3":
        cfg = TransformerConfig(**{**{f.name: getattr(cfg, f.name) for f in __import__("dataclasses").fields(cfg) if f.init}, **dict(
            num_moe_experts=8, moe_router_topk=4, moe_router_score_function="sigmoid", moe_router_num_groups=2, moe_router_group_topk=1, moe_router_topk_scaling_factor=2.5,
            moe_router_load_balancing_type="seq_aux_loss", moe_aux_loss_coeff=0.01, moe_z_loss_coeff=1e-3, moe_shared_expert_intermediate_size=64, moe_ffn_hidden_size=48,
            moe_router_pre_softmax=False), **__import__("json").loads(os.environ.get("REF_MOE_OVERRIDE", "{}"))})
    if variant == "moe_drop":
        cfg = TransformerConfig(**{**{f.name: getattr(cfg, f.name) for f in __import__("dataclasses").fields(cfg) if f.init}, **dict(
            moe_token_dispatcher_type="alltoall", moe_expert_capacity_factor=1.0, moe_token_drop_policy="probs", moe_pad_expert_input_to_capacity=True, moe_router_pre_softmax=True)})
    spec = get_gpt_layer_local_spec(num_experts=cfg.num_moe_experts, moe_grouped_gemm=False, normalization="RMSNorm") if variant.startswith("moe") else get_gpt_layer_local_spec(normalization="RMSNorm")
    m = GPTModel(cfg, spec, vocab_size=CFG["vocab"], max_sequence_length=CFG["seq"], parallel_output=True,
                 share_embeddings_and_output_weights=False, position_embedding_type="rope", rotary_base=10000)
    with torch.no_grad():
        for n, p in m.named_parameters():
            if p.dim() == 1:
                p.fill_(1.0)
                continue
            sharded = bool(getattr(p, "tensor_model_parallel", False)) and tp > 1
            dim = int(getattr(p, "partition_dim", -1))
            shape = list(p.shape)
            if sharded:
                shape[dim] *= tp
            g = torch.Generator().manual_seed(zlib.crc32(n.encode()))
            full = torch.empty(shape).normal_(0, 0.05, generator=g)
            r = ps.get_tensor_model_parallel_rank()
            if sharded and n.endswith("linear_fc1.weight"):
                ga, up = full.chunk(2, dim=0)
                p.copy_(torch.cat([ga.chunk(tp, dim=0)[r], up.chunk(tp, dim=0)[r]], dim=0))
            else:
                p.copy_(full.chunk(tp, dim=dim)[r] if sharded else full)
    tok = torch.randint(0, CFG["vocab"], (CFG["batch"], CFG["seq"] + 1), generator=torch.Generator().manual_seed(1))
    if ep2:
        tok = tok[rank:rank + 1]
    pos = torch.arange(CFG["seq"]).unsqueeze(0).expand(tok.shape[0], -1).contiguous()
    loss = m(tok[:, :-1].contiguous(), pos, None, labels=tok[:, 1:].contiguous()).float().mean()
    loss.backward()
    return {"loss": float(loss), "grads": {n: p.grad.clone() for n, p in m.named_parameters()}, "names": [n for n, _ in m.named_parameters()]}


@pytest.mark.parametrize("tp", [1, 2])
def test_loss_and_grad_parity_with_reference(tmp_path, tp):
    from dist_utils import run_distributed

    ref = _reference(f"gpt_tp{tp}")
    ours = run_distributed(_ours, tp, tp)
    for r in range(tp):
        assert sorted(ours[r]["names"]) == sorted(ref[r]["grads"].keys()), "parameter names differ from the reference's"
        assert abs(ours[r]["loss"] - ref[r]["loss"]) < 2e-5, (ours[r]["loss"], ref[r]["loss"])
        _assert_tensors_match(ours[r]["grads"], ref[r]["grads"], 2e-4, f"rank {r} grad")


def test_moe_loss_and_grad_parity_with_reference(tmp_path):
    """A 4-expert top-2 MoE GPT (router + aux loss, all-gather dispatcher, per-expert MLPs): same parameter names, loss and gradients as the unmodified reference."""
    from dist_utils import run_distributed

    ref = _reference("moe")[0]
    ours = run_distributed(_ours, 1, 1, "moe")[0]
    assert sorted(ours["names"]) == sorted(ref["grads"].keys()), (sorted(set(ours["names"]) ^ set(ref["grads"].keys())))
    assert any("router" in n for n in ours["names"]) and any("local_experts" in n for n in ours["names"])
    assert abs(ours["loss"] - ref["loss"]) < 2e-5, (ours["loss"], ref["loss"])
    _assert_tensors_match(ours["grads"], ref["grads"], 5e-4, "grad")


def test_moe_deepseek_style_router_parity_with_reference(tmp_path):
    """8 experts, top-4 from 1 of 2 groups, sigmoid scores with a scaling factor, per-sequence aux loss, z-loss, a shared expert: names, loss and gradients equal the
    unmodified reference's."""
    from dist_utils import run_distributed

    ref = _reference("moe_dsv3")[0]
    ours = run_distributed(_ours, 1, 1, "moe_dsv3")[0]
    assert sorted(ours["names"]) == sorted(ref["grads"].keys()), sorted(set(ours["names"]) ^ set(ref["grads"].keys()))
    assert any("shared_experts" in n for n in ours["names"])
    assert abs(ours["loss"] - ref["loss"]) < 2e-5, (ours["loss"], ref["loss"])
    _assert_tensors_match(ours["grads"], ref["grads"], 1e-3, "grad")


def test_moe_capacity_drop_and_pad_parity_with_reference(tmp_path):
    """Capacity factor 1.0 with probability-based token dropping and padding to capacity (all-to-all dispatcher): the same tokens are dropped, the loss and every
    gradient equal the unmodified reference's."""
    from dist_utils import run_distributed

    ref = _reference("moe_drop")[0]
    ours = run_distributed(_ours, 1, 1, "moe_drop")[0]
    assert sorted(ours["names"]) == sorted(ref["grads"].keys())
    assert abs(ours["loss"] - ref["loss"]) < 2e-5, (ours["loss"], ref["loss"])
    _assert_tensors_match(ours["grads"], ref["grads"], 1e-3, "grad")


def test_mup_parity_with_reference(tmp_path, monkeypatch):
    """Maximal-update parametrisation on (width multiplier 2, embedding multiplier 2): attention scaled by 1/d_head, embeddings and logits multiplied — the
    loss and every gradient equal the unmodified reference's; and the run differs from the plain one (the switch is not a no-op)."""
    from dist_utils import run_distributed

    plain = run_distributed(_ours, 1, 1, "")[0]
    monkeypatch.setenv("REF_CFG_OVERRIDE", '{"use_mup": true, "mup_base_hidden_size": 32, "mup_embedding_mult": 2.0}')
    ref = _reference("mup")[0]
    ours = run_distributed(_ours, 1, 1, "")[0]
    assert abs(ours["loss"] - plain["loss"]) > 1e-3
    assert abs(ours["loss"] - ref["loss"]) < 2e-5, (ours["loss"], ref["loss"])
    _assert_tensors_match(ours["grads"], ref["grads"], 1e-3, "grad")


def test_moe_expert_parallel_parity_with_reference(tmp_path):
    """Expert parallel 2 over gloo (2 of the 4 experts per rank, each rank feeds its own half of the batch; the all-gather dispatcher — the reference's all-to-all
    dispatcher passes tensor split sizes that gloo rejects): per-rank loss and gradients, incl. the expert weights that received tokens from the OTHER rank,
    equal the unmodified reference's."""
    from dist_utils import run_distributed

    ref = _reference("moe_ep2")
    ours = run_distributed(_ours, 2, 1, "moe_ep2")
    for r in range(2):
        assert sorted(ours[r]["names"]) == sorted(ref[r]["grads"].keys())
        assert abs(ours[r]["loss"] - ref[r]["loss"]) < 2e-5, (r, ours[r]["loss"], ref[r]["loss"])
        _assert_tensors_match(ours[r]["grads"], ref[r]["grads"], 5e-4, f"rank {r} grad")


def _ours_bert(rank, world):
    import zlib

    from megatron_b200.core import parallel_state as ps
    from megatron_b200.core.models.bert.bert_layer_specs import bert_layer_local_spec
    from megatron_b200.core.models.bert.bert_model import BertModel
    from megatron_b200.core.transformer.transformer_config import TransformerConfig

    ps.initialize_model_parallel()
    cfg = TransformerConfig(num_layers=2, hidden_size=64, ffn_hidden_size=128, num_attention_heads=4, hidden_dropout=0.0, attention_dropout=0.0, use_cpu_initialization=True,
                            gradient_accumulation_fusion=False, perform_initialization=False, layernorm_epsilon=1e-5, bias_dropout_fusion=False)
    m = BertModel(cfg, num_tokentypes=2, transformer_layer_spec=bert_layer_local_spec, vocab_size=128, max_sequence_length=32, parallel_output=True, add_binary_head=True)

    def seeded(n, shape, std):
        return torch.empty(shape).normal_(0, std, generator=torch.Generator().manual_seed(zlib.crc32(n.encode())))

    with torch.no_grad():
        for n, p in m.named_parameters():
            if p.dim() == 1:
                p.copy_(seeded(n, list(p.shape), 0.02)) if "bias" in n else p.fill_(1.0)
            else:
                p.copy_(seeded(n, list(p.shape), 0.05))
    g = torch.Generator().manual_seed(3)
    tok = torch.randint(0, 128, (2, 32), generator=g)
    types = torch.randint(0, 2, (2, 32), generator=g)
    pad = torch.ones(2, 32, dtype=torch.long)
    pad[1, 25:] = 0
    labels = torch.randint(0, 128, (2, 32), generator=g)
    lm_loss, binary = m(tok, pad, tokentype_ids=types, lm_labels=labels)
    loss = (lm_loss.float() * pad).sum() / pad.sum() + binary.float().logsumexp(-1).mean()
    loss.backward()
    return {"loss": float(loss), "grads": {n: p.grad.clone() for n, p in m.named_parameters() if p.grad is not None}, "names": [n for n, p in m.named_parameters() if p.grad is not None]}


def test_bert_parity_with_reference(tmp_path):
    """BERT (token types, learned positions, padding mask, LM head, pooler + binary head): parameter names, loss and gradients equal the unmodified reference's."""
    from dist_utils import run_distributed

    ref = _reference("bert")[0]
    ours = run_distributed(_ours_bert, 1)[0]
    assert sorted(ours["names"]) == sorted(ref["grads"].keys()), sorted(set(ours["names"]) ^ set(ref["grads"].keys()))
    assert abs(ours["loss"] - ref["loss"]) < 2e-5, (ours["loss"], ref["loss"])
    _assert_tensors_match(ours["grads"], ref["grads"], 5e-4, "grad")


def _ours_t5(rank, world):
    import zlib

    sys.path.insert(0, os.path.join(REPO, "tests", "helpers"))
    from megatron_b200.core import parallel_state as ps
    from megatron_b200.core.models.T5.t5_model import T5Model
    from megatron_b200.core.models.T5.t5_spec import get_t5_decoder_with_local_block_spec, get_t5_encoder_with_local_block_spec
    from megatron_b200.core.transformer.transformer_config import TransformerConfig

    ps.initialize_model_parallel()
    kw = dict(hidden_size=64, ffn_hidden_size=128, num_attention_heads=4, kv_channels=16, hidden_dropout=0.0, attention_dropout=0.0, use_cpu_initialization=True,
              gradient_accumulation_fusion=False, perform_initialization=False, bias_dropout_fusion=False)
    cfg, enc_cfg = TransformerConfig(num_layers=2, **kw), TransformerConfig(num_layers=2, **kw)
    # the TE-less reference resolves the block's ``layer_norm=TENorm`` to nothing (no final layer norms); build the same structure here
    enc_spec, dec_spec = get_t5_encoder_with_local_block_spec(2), get_t5_decoder_with_local_block_spec(2)
    enc_spec.layer_norm = dec_spec.layer_norm = None
    m = T5Model(cfg, enc_cfg, enc_spec, dec_spec, vocab_size=128, max_sequence_length=32, parallel_output=True, share_embeddings_and_output_weights=True)

    def seeded(n, shape, std):
        return torch.empty(shape).normal_(0, std, generator=torch.Generator().manual_seed(zlib.crc32(n.encode())))

    with torch.no_grad():
        for n, p in m.named_parameters():
            if p.dim() == 1:
                p.copy_(seeded(n, list(p.shape), 0.02)) if "bias" in n else p.fill_(1.0)
            else:
                p.copy_(seeded(n, list(p.shape), 0.05))
    g = torch.Generator().manual_seed(5)
    b, se, sd = 2, 24, 12
    enc = torch.randint(0, 128, (b, se), generator=g)
    dec = torch.randint(0, 128, (b, sd), generator=g)
    labels = torch.randint(0, 128, (b, sd), generator=g)
    enc_keep = torch.ones(b, se)
    enc_keep[1, 20:] = 0
    enc_mask = enc_keep[:, :, None] * enc_keep[:, None, :]
    dec_mask = torch.tril(torch.ones(sd, sd))[None].expand(b, -1, -1).contiguous()
    x_mask = torch.ones(b, sd, 1) * enc_keep[:, None, :]
    # the reference's calling convention: already-extended boolean masks, True = masked
    loss = m(enc, dec, (enc_mask < 0.5).unsqueeze(1), (dec_mask < 0.5).unsqueeze(1), (x_mask < 0.5).unsqueeze(1), lm_labels=labels).float().mean()
    loss.backward()
    loss2 = m(enc, dec, enc_mask, dec_mask, x_mask, lm_labels=labels).float().mean()             # this framework's keep-mask convention gives the same result
    assert abs(float(loss2) - float(loss)) < 1e-6
    return {"loss": float(loss), "grads": {n: p.grad.clone() for n, p in m.named_parameters() if p.grad is not None}, "names": [n for n, p in m.named_parameters() if p.grad is not None]}


def test_t5_parity_with_reference(tmp_path):
    """T5 encoder-decoder (cross attention, padding / causal / cross masks, shared embeddings + LM-head bias): names, loss and gradients equal the reference's."""
    from dist_utils import run_distributed

    ref = _reference("t5")[0]
    ours = run_distributed(_ours_t5, 1)[0]
    assert sorted(ours["names"]) == sorted(ref["grads"].keys()), sorted(set(ours["names"]) ^ set(ref["grads"].keys()))
    assert abs(ours["loss"] - ref["loss"]) < 2e-5, (ours["loss"], ref["loss"])
    _assert_tensors_match(ours["grads"], ref["grads"], 5e-4, "grad")


def _ours_vit(rank, world):
    import zlib

    from megatron_b200.core import parallel_state as ps
    from megatron_b200.core.models.vision.clip_vit_model import CLIPViTModel
    from megatron_b200.core.models.vision.vit_layer_specs import get_vit_layer_with_local_spec
    from megatron_b200.core.transformer.torch_norm import FusedNorm
    from megatron_b200.core.transformer.transformer_config import TransformerConfig

    ps.initialize_model_parallel()
    cfg = TransformerConfig(num_layers=2, hidden_size=64, ffn_hidden_size=128, num_attention_heads=4, hidden_dropout=0.0, attention_dropout=0.0, use_cpu_initialization=True,
                            gradient_accumulation_fusion=False, perform_initialization=False, bias_dropout_fusion=False)
    m = CLIPViTModel(cfg, get_vit_layer_with_local_spec(), ln_pre_impl=FusedNorm, ln_post_impl=FusedNorm, patch_dim=14, img_h=28, img_w=28)

    def seeded(n, shape, std):
        return torch.empty(shape).normal_(0, std, generator=torch.Generator().manual_seed(zlib.crc32(n.encode())))

    with torch.no_grad():
        for n, p in m.named_parameters():
            if p.dim() == 1:
                p.copy_(seeded(n, list(p.shape), 0.02)) if "bias" in n else p.fill_(1.0)
            else:
                p.copy_(seeded(n, list(p.shape), 0.05))
    x = torch.randn(2, 3, 28, 28, generator=torch.Generator().manual_seed(7))
    out = m(x)
    w = torch.randn(out.shape, generator=torch.Generator().manual_seed(8))
    loss = (out.float() * w).mean()
    loss.backward()
    return {"loss": float(loss), "shape": tuple(out.shape), "grads": {n: p.grad.clone() for n, p in m.named_parameters() if p.grad is not None},
            "names": [n for n, p in m.named_parameters() if p.grad is not None]}


def test_clip_vit_parity_with_reference(tmp_path):
    """CLIP ViT tower (conv patch embedding, class token, learned positions, pre-norm): output shape, parameter names, loss and gradients equal the reference's."""
    from dist_utils import run_distributed

    ref = _reference("vit")[0]
    ours = run_distributed(_ours_vit, 1)[0]
    assert list(ours["shape"]) == ref["shape"]
    assert sorted(ours["names"]) == sorted(ref["grads"].keys()), sorted(set(ours["names"]) ^ set(ref["grads"].keys()))
    assert abs(ours["loss"] - ref["loss"]) < 1e-6, (ours["loss"], ref["loss"])
    _assert_tensors_match(ours["grads"], ref["grads"], 5e-4, "grad")


def _ours_optim(rank, world, dist_opt=False):
    sys.path.insert(0, os.path.join(REPO, "tests", "helpers"))
    from megatron_b200.core.distributed import DistributedDataParallel, DistributedDataParallelConfig
    from megatron_b200.core.optimizer import OptimizerConfig, get_megatron_optimizer
    from megatron_b200.core.optimizer_param_scheduler import OptimizerParamScheduler

    m, _ = _our_model(1)
    _seeded_init(m, 0, 1)
    cfg = m.config
    m = DistributedDataParallel(cfg, DistributedDataParallelConfig(grad_reduce_in_fp32=True, overlap_grad_reduce=False, use_distributed_optimizer=dist_opt), m)
    ocfg = OptimizerConfig(optimizer="adam", lr=1e-2, min_lr=1e-3, weight_decay=0.1, adam_beta1=0.9, adam_beta2=0.95, adam_eps=1e-8, clip_grad=0.5, bf16=False, fp16=False,
                           use_distributed_optimizer=dist_opt)
    opt = get_megatron_optimizer(ocfg, [m])
    sched = OptimizerParamScheduler(opt, init_lr=0.0, max_lr=1e-2, min_lr=1e-3, lr_warmup_steps=2, lr_decay_steps=10, lr_decay_style="cosine", start_wd=0.1, end_wd=0.1,
                                    wd_incr_steps=10, wd_incr_style="constant")
    tok = torch.randint(0, 128, (2, 33), generator=torch.Generator().manual_seed(1))
    if dist_opt:
        tok = tok[rank:rank + 1]
    pos = torch.arange(32).unsqueeze(0).expand(tok.shape[0], -1).contiguous()
    losses, norms = [], []
    for it in range(3):
        m.zero_grad_buffer()
        opt.zero_grad()
        loss = m(tok[:, :-1].contiguous(), pos, None, labels=tok[:, 1:].contiguous()).float().mean()
        loss.backward()
        m.finish_grad_sync()
        ok, gn, _ = opt.step()
        sched.step(increment=1)
        losses.append(float(loss))
        norms.append(float(gn))
    return {"losses": losses, "grad_norms": norms, "lr": [g["lr"] for g in opt.param_groups], "params": {n: p.detach().clone() for n, p in m.module.named_parameters()}}


def test_optimizer_stack_parity_with_reference(tmp_path):
    """Three training steps through DDP + the optimizer stack + the LR / WD scheduler (param groups with and without weight decay, global-norm clipping at 0.5,
    warm-up from 0 then cosine decay): losses, gradient norms, learning rates and the final parameters equal the unmodified reference's."""
    from dist_utils import run_distributed

    ref = _reference("optim")[0]
    ours = run_distributed(_ours_optim, 1)[0]
    assert all(abs(a - b) < 2e-5 for a, b in zip(ours["losses"], ref["losses"])), (ours["losses"], ref["losses"])
    assert all(abs(a - b) < 1e-4 * b for a, b in zip(ours["grad_norms"], ref["grad_norms"])), (ours["grad_norms"], ref["grad_norms"])
    assert sorted(round(x, 9) for x in ours["lr"]) == sorted(round(x, 9) for x in ref["lr"]), (ours["lr"], ref["lr"])
    assert ours["losses"][2] < ours["losses"][0]
    _assert_tensors_match(ours["params"], ref["params"], 2e-5, "param after 3 steps", relative=False)


def test_distributed_optimizer_parity_with_reference(tmp_path):
    """Data parallel 2 over gloo with the distributed (ZeRO-1) optimizer: reduce-scattered gradients, sharded Adam state, parameter all-gather — per-rank losses,
    the global gradient norm and every rank's parameters after three steps equal the unmodified reference's."""
    from dist_utils import run_distributed

    ref = _reference("distopt")
    ours = run_distributed(_ours_optim, 2, True)
    for r in range(2):
        assert all(abs(a - b) < 2e-5 for a, b in zip(ours[r]["losses"], ref[r]["losses"])), (r, ours[r]["losses"], ref[r]["losses"])
        assert all(abs(a - b) < 1e-4 * b for a, b in zip(ours[r]["grad_norms"], ref[r]["grad_norms"])), (ours[r]["grad_norms"], ref[r]["grad_norms"])
        _assert_tensors_match(ours[r]["params"], ref[r]["params"], 2e-5, f"rank {r} param after 3 steps", relative=False)
    assert all(torch.equal(ours[0]["params"][n], ours[1]["params"][n]) for n in ours[0]["params"])        # replicas stay in sync


def _ours_pp2(rank, world):
    import zlib

    import torch.nn.functional as F

    from megatron_b200.core import parallel_state as ps
    from megatron_b200.core.models.gpt.gpt_layer_specs import get_gpt_layer_local_spec
    from megatron_b200.core.models.gpt.gpt_model import GPTModel
    from megatron_b200.core.pipeline_parallel import get_forward_backward_func
    from megatron_b200.core.transformer.transformer_config import TransformerConfig

    ps.initialize_model_parallel(pipeline_model_parallel_size=2)
    pre, post = ps.is_pipeline_first_stage(), ps.is_pipeline_last_stage()
    cfg = TransformerConfig(num_layers=4, hidden_size=64, ffn_hidden_size=128, num_attention_heads=4, num_query_groups=2, kv_channels=16, normalization="RMSNorm",
                            gated_linear_unit=True, activation_func=F.silu, add_bias_linear=False, hidden_dropout=0.0, attention_dropout=0.0, use_cpu_initialization=True,
                            gradient_accumulation_fusion=False, perform_initialization=False, pipeline_model_parallel_size=2, pipeline_dtype=torch.float32, bias_dropout_fusion=False)
    m = GPTModel(cfg, get_gpt_layer_local_spec(normalization="RMSNorm"), vocab_size=128, max_sequence_length=32, pre_process=pre, post_process=post, parallel_output=True,
                 share_embeddings_and_output_weights=False, position_embedding_type="rope", rotary_base=10000)
    off = 0 if pre else 2
    with torch.no_grad():
        for n, p in m.named_parameters():
            gname = n
            if ".layers." in n:
                head, rest = n.split(".layers.")
                i, tail = rest.split(".", 1)
                gname = f"{head}.layers.{int(i) + off}.{tail}"
            if p.dim() == 1:
                p.fill_(1.0)
            else:
                p.copy_(torch.empty(list(p.shape)).normal_(0, 0.05, generator=torch.Generator().manual_seed(zlib.crc32(gname.encode()))))
    toks = torch.randint(0, 128, (4, 2, 33), generator=torch.Generator().manual_seed(2))
    pos = torch.arange(32).unsqueeze(0).expand(2, -1).contiguous()

    def loss_func(output):
        loss = output.float().mean()
        return loss, {"lm loss": loss.detach().clone()}

    def forward_step(data_iterator, model):
        t = next(data_iterator)
        return model(t[:, :-1].contiguous(), pos, None, labels=t[:, 1:].contiguous()), loss_func

    out = get_forward_backward_func()(forward_step_func=forward_step, data_iterator=iter(toks), model=[m], num_microbatches=4, seq_length=32, micro_batch_size=2, forward_only=False)
    losses = [float(d["lm loss"]) for d in out] if post else []
    return {"losses": losses, "grads": {n: p.grad.clone() for n, p in m.named_parameters() if p.grad is not None}}


def test_pipeline_schedule_parity_with_reference(tmp_path):
    """Pipeline parallel 2 over gloo, 1F1B with 4 micro-batches: the per-micro-batch losses on the last stage and every stage's accumulated gradients equal the
    unmodified reference's schedule (same loss scaling by the number of micro-batches, same p2p tensor flow)."""
    from dist_utils import run_distributed

    ref = _reference("pp2")
    ours = run_distributed(_ours_pp2, 2)
    assert ours[0]["losses"] == [] and len(ours[1]["losses"]) == 4
    assert all(abs(a - b) < 2e-5 for a, b in zip(ours[1]["losses"], ref[1]["losses"])), (ours[1]["losses"], ref[1]["losses"])
    for r in range(2):
        assert sorted(ours[r]["grads"]) == sorted(ref[r]["grads"]), (r, sorted(set(ours[r]["grads"]) ^ set(ref[r]["grads"])))
        _assert_tensors_match(ours[r]["grads"], ref[r]["grads"], 5e-4, f"stage {r} grad")


# ---- distributed-checkpoint interop (SURVEY 7.4-6: "cross-load a checkpoint with the reference") --------------------------------------


# The interop model is smaller than the parity model so that the reference's checkpoints of it can be stored (keys of ``CFG`` in ref_cpu_model.py).
CKPT_MODEL = dict(hidden_size=16, ffn_hidden_size=32, kv_channels=4, vocab=32, seq=8)


def _reference_checkpoint(tmp_path, tp):
    """Unpack the reference's checkpoint written at TP=tp."""
    import tarfile

    dst = tmp_path / f"ckpt_ref_tp{tp}"
    with tarfile.open(os.path.join(GOLDEN, f"ckpt_tp{tp}.tar.gz")) as tar:
        tar.extractall(dst, filter="data")
    return dst


def _dcp_tensors(ckpt_dir):
    """Every tensor of a torch_dist checkpoint, read in full by torch.distributed.checkpoint (the reader both frameworks load through)."""
    import torch.distributed.checkpoint as dcp
    from torch.distributed.checkpoint.metadata import TensorStorageMetadata

    md = dcp.FileSystemReader(str(ckpt_dir)).read_metadata()
    sd = {k: torch.empty(list(m.size), dtype=m.properties.dtype) for k, m in md.state_dict_metadata.items() if isinstance(m, TensorStorageMetadata)}
    dcp.load(sd, storage_reader=dcp.FileSystemReader(str(ckpt_dir)), no_dist=True)
    return sd


def _our_model(tp, num_layers=2, hidden_size=64, ffn_hidden_size=128, num_attention_heads=4, num_query_groups=2, kv_channels=16, vocab=128, seq=32):
    import torch.nn.functional as F

    from megatron_b200.core import parallel_state as ps
    from megatron_b200.core.models.gpt.gpt_layer_specs import get_gpt_layer_local_spec
    from megatron_b200.core.models.gpt.gpt_model import GPTModel
    from megatron_b200.core.transformer.transformer_config import TransformerConfig

    ps.initialize_model_parallel(tensor_model_parallel_size=tp)
    cfg = TransformerConfig(num_layers=num_layers, hidden_size=hidden_size, ffn_hidden_size=ffn_hidden_size, num_attention_heads=num_attention_heads,
                            num_query_groups=num_query_groups, kv_channels=kv_channels, normalization="RMSNorm",
                            gated_linear_unit=True, activation_func=F.silu, add_bias_linear=False, hidden_dropout=0.0, attention_dropout=0.0, use_cpu_initialization=True,
                            gradient_accumulation_fusion=False, perform_initialization=False, tensor_model_parallel_size=tp)
    m = GPTModel(cfg, get_gpt_layer_local_spec(normalization="RMSNorm"), vocab_size=vocab, max_sequence_length=seq, parallel_output=True,
                 share_embeddings_and_output_weights=False, position_embedding_type="rope", rotary_base=10000)
    return m, ps.get_tensor_model_parallel_rank()


def _seeded_init(m, tp_rank, tp):
    import zlib

    with torch.no_grad():
        for n, p in m.named_parameters():
            if p.dim() == 1:
                p.fill_(1.0)
                continue
            sharded = bool(getattr(p, "tensor_model_parallel", False)) and tp > 1
            dim = int(getattr(p, "partition_dim", -1))
            shape = list(p.shape)
            if sharded:
                shape[dim] *= tp
            g = torch.Generator().manual_seed(zlib.crc32(n.encode()))
            full = torch.empty(shape).normal_(0, 0.05, generator=g)
            if sharded and n.endswith("linear_fc1.weight"):
                ga, up = full.chunk(2, dim=0)
                p.copy_(torch.cat([ga.chunk(tp, dim=0)[tp_rank], up.chunk(tp, dim=0)[tp_rank]], dim=0))
            else:
                p.copy_(full.chunk(tp, dim=dim)[tp_rank] if sharded else full)


def _ours_save(rank, world, tp, ckpt_dir):
    from megatron_b200.core import dist_checkpointing

    m, tp_rank = _our_model(tp, **CKPT_MODEL)
    _seeded_init(m, tp_rank, tp)
    dist_checkpointing.save(m.sharded_state_dict(), ckpt_dir)
    return True


def _ours_load(rank, world, tp, ckpt_dir):
    from megatron_b200.core import dist_checkpointing

    m, tp_rank = _our_model(tp, **CKPT_MODEL)
    with torch.no_grad():
        for _, p in m.named_parameters():
            p.zero_()
    sd = dist_checkpointing.load(m.sharded_state_dict(), ckpt_dir)
    m.load_state_dict(sd, strict=False)
    got = {n: p.detach().clone() for n, p in m.named_parameters()}
    _seeded_init(m, tp_rank, tp)
    return max(float((got[n] - p.detach()).abs().max()) for n, p in m.named_parameters())


@pytest.mark.parametrize("tp_write,tp_read", [(2, 1), (1, 2)])
def test_reference_loads_our_checkpoint(tmp_path, tp_write, tp_read):
    """A torch_dist checkpoint written by this framework (TP=tp_write) holds, under every key and global shape of the UNMODIFIED reference's own checkpoint
    of the same model at TP=tp_read, exactly the tensors the reference wrote there: what the reference reads back at that TP size."""
    from dist_utils import run_distributed

    ckpt = tmp_path / "ckpt_ours"
    ckpt.mkdir()
    run_distributed(_ours_save, tp_write, tp_write, str(ckpt))
    ours, ref = _dcp_tensors(ckpt), _dcp_tensors(_reference_checkpoint(tmp_path, tp_read))
    assert sorted(ours) == sorted(ref) and len(ref) > 0, sorted(set(ours) ^ set(ref))
    for k, t in ref.items():
        assert ours[k].dtype == t.dtype and torch.equal(ours[k], t), k


@pytest.mark.parametrize("tp_write,tp_read", [(2, 1), (1, 2)])
def test_we_load_reference_checkpoint(tmp_path, tp_write, tp_read):
    """...and a checkpoint written by the reference (stored) is read by this framework, resharded."""
    from dist_utils import run_distributed

    ckpt = _reference_checkpoint(tmp_path, tp_write)
    diffs = run_distributed(_ours_load, tp_read, tp_read, str(ckpt))
    assert all(d == 0.0 for d in diffs), diffs


# ---- data pipeline -----------------------------------------------------------------------------------------------------------------------------


DATA_SEQ, DATA_SEED, DATA_SPLIT, DATA_COUNTS = 32, 1234, "80,15,5", [64, 12, 8]


def _write_corpus(prefix, n_docs, seed):
    import numpy as np

    from megatron_b200.core.datasets.indexed_dataset import IndexedDatasetBuilder

    rng = np.random.default_rng(seed)
    b = IndexedDatasetBuilder(prefix + ".bin", dtype=np.int32)
    for _ in range(n_docs):
        doc = rng.integers(1, 99, size=int(rng.integers(3, 60))).tolist() + [99]
        b.add_document(np.asarray(doc, dtype=np.int32), [len(doc)])
    b.finalize(prefix + ".idx")


def write_corpora(d):
    _write_corpus(os.path.join(d, "a"), 300, 1)
    _write_corpus(os.path.join(d, "b"), 200, 2)


def data_blend_args(d, blend):
    return ["0.7", os.path.join(d, "a"), "0.3", os.path.join(d, "b")] if blend else ["1.0", os.path.join(d, "a")]


@pytest.mark.parametrize("blend", [False, True])
def test_gpt_dataset_samples_match_reference(tmp_path, blend):
    """The reference read the .bin/.idx files THIS framework writes, and both build the same train / valid / test samples from them (document shuffle, sample
    index, blending of two corpora, loss masks, reset position ids) for the same seed — a run switched over sees the same data order."""
    from megatron_b200.core.datasets import BlendedMegatronDatasetBuilder, GPTDatasetConfig
    from megatron_b200.core.datasets.gpt_dataset import GPTDataset
    from megatron_b200.core.datasets.utils import get_blend_from_list

    write_corpora(str(tmp_path))
    blend_args = data_blend_args(str(tmp_path), blend)
    with open(os.path.join(GOLDEN, f"gpt_dataset_{'blend' if blend else 'single'}.json")) as f:
        ref = json.load(f)

    class Tok:
        eod = 99
        unique_identifiers = {"class": "TestTokenizer", "eod": 99}

    cfg = GPTDatasetConfig(random_seed=DATA_SEED, sequence_length=DATA_SEQ, blend=get_blend_from_list(blend_args), split=DATA_SPLIT, path_to_cache=str(tmp_path / "our_cache"),
                           tokenizer=Tok(), reset_position_ids=True, reset_attention_mask=False, eod_mask_loss=True, create_attention_mask=False, mmap_bin_files=False)
    ours = BlendedMegatronDatasetBuilder(GPTDataset, DATA_COUNTS, lambda: True, cfg).build()
    for name, ds in zip(("train", "valid", "test"), ours):
        assert (ds is None) == (ref[name] is None)
        if ds is None:
            continue
        assert len(ds) == ref[name]["len"], (name, len(ds), ref[name]["len"])
        for i, want in ref[name]["samples"].items():
            got = ds[int(i)]
            for k, (dtype, values) in want.items():
                v = torch.tensor(values, dtype=getattr(torch, dtype))
                assert torch.equal(torch.as_tensor(got[k]).to(v.dtype), v), (name, i, k)


# ---- pure-Python subsystems: schedules, micro-batch ramp-up, rank enumeration ------------------------------------------------------------
@pytest.fixture(scope="module")
def ref_pure():
    with open(os.path.join(GOLDEN, "schedules_and_ranks.json")) as f:
        return json.load(f)


def _pure_cfg():
    import importlib.util

    spec = importlib.util.spec_from_file_location("_ref_pure_cfg", os.path.join(REPO, "tests", "helpers", "ref_pure.py"))
    src = open(spec.origin).read().split("class _Opt")[0].split("SCHEDULES = ")[1]
    ns = {}
    exec("SCHEDULES = " + src, ns)
    return ns


def test_lr_wd_schedules_match_reference(ref_pure):
    from megatron_b200.core.optimizer_param_scheduler import OptimizerParamScheduler

    cfg = _pure_cfg()

    class Opt:
        def __init__(self):
            self.param_groups = [{"lr": 0.0, "weight_decay": 0.0, "lr_mult": 1.0, "wd_mult": 1.0},
                                 {"lr": 0.0, "weight_decay": 0.0, "wd_mult": 0.5, "max_lr": 5e-4, "min_lr": 5e-5, "start_wd": 0.2, "end_wd": 0.2}]

    for kw, want in zip(cfg["SCHEDULES"], ref_pure["sched"]):
        opt = Opt()
        s = OptimizerParamScheduler(opt, **kw)
        for step, row in enumerate(want):
            s.step(increment=1)
            got = [[g["lr"], g["weight_decay"]] for g in opt.param_groups]
            for (glr, gwd), (rlr, rwd) in zip(got, row):
                assert glr == pytest.approx(rlr, rel=1e-12, abs=1e-18), (kw["lr_decay_style"], step)
                assert gwd == pytest.approx(rwd, rel=1e-12, abs=1e-18), (kw["wd_incr_style"], step)


def test_microbatch_schedules_match_reference(ref_pure):
    from megatron_b200.core.num_microbatches_calculator import (destroy_num_microbatches_calculator, get_current_global_batch_size, get_num_microbatches,
                                                                 init_num_microbatches_calculator, update_num_microbatches)

    cfg = _pure_cfg()
    for kw, want in zip(cfg["RAMPS"], ref_pure["ramp"]):
        destroy_num_microbatches_calculator()
        init_num_microbatches_calculator(rank=0, **kw)
        got = []
        for consumed in range(0, 320, 8):
            update_num_microbatches(consumed, consistency_check=False)
            got.append([get_num_microbatches(), get_current_global_batch_size()])
        destroy_num_microbatches_calculator()
        assert got == want, kw


def test_rank_generator_matches_reference(ref_pure):
    from megatron_b200.core.parallel_state import RankGenerator

    cfg = _pure_cfg()
    for kw, want in zip(cfg["GRIDS"], ref_pure["ranks"]):
        g = RankGenerator(**kw)
        for tok in cfg["TOKENS"]:
            if isinstance(want[tok], str):
                continue
            assert g.get_ranks(tok) == want[tok], (kw, tok)
