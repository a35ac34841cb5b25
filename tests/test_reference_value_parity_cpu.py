"""DSA mask / indexer-loss helpers, MoE routing scores and hybrid layer patterns: value parity with the unmodified reference's pure-PyTorch functions.

Each ``_*_outputs(mod)`` evaluates one module on fixed, seeded inputs.  The reference's results for the same calls are stored in
``tests/golden/reference/value_parity.pt`` (written by ``tests/helpers/make_reference_golden.py``); the tests run this framework's module and
compare."""
import os

import pytest
import torch

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference", "value_parity.pt")


def _golden(name):
    return torch.load(GOLDEN)[name]


def _indexer_inputs():
    torch.manual_seed(0)
    target = torch.rand(2, 5, 7) * (torch.rand(2, 5, 7) > 0.3)
    target[0, 1] = 0                                                    # a row without any mass
    valid = torch.rand(2, 5, 7) > 0.2
    logp = torch.log_softmax(torch.randn(2, 5, 7), -1).masked_fill(~valid, float("-inf"))
    rows = torch.rand(2, 5) > 0.3
    return target, valid, logp, rows


def _indexer_loss_outputs(M):
    target, valid, logp, rows = _indexer_inputs()
    t = M.normalize_indexer_target(target)
    out = {"target": t, "kl_per_row": M.indexer_kl_per_row(t, logp, valid)}
    for per_token in (False, True):
        for qv_name, qv in (("all", None), ("rows", rows)):
            out[f"loss_{per_token}_{qv_name}"] = M.indexer_loss_from_target(t, logp, 0.3, qv, per_token, valid)
    return out


def test_indexer_loss_matches_reference():
    from megatron_b200.core.transformer.experimental_attention_variant import dsa_indexer_loss as M

    want = _golden("dsa_indexer_loss")
    got = _indexer_loss_outputs(M)
    assert sorted(got) == sorted(want)
    assert torch.allclose(got["target"], want["target"])
    assert torch.allclose(got["kl_per_row"], want["kl_per_row"])
    for k in got:
        if k.startswith("loss_"):
            assert torch.isfinite(got[k]) and torch.allclose(got[k], want[k]), k
    target = _indexer_inputs()[0]
    assert torch.equal(M.normalize_indexer_target_(target.clone()), got["target"])


def _masking_outputs(M, device):
    torch.manual_seed(1)
    cu = torch.tensor([0, 3, 3, 9, 12], dtype=torch.int32)             # incl. an empty sequence
    s, e = M.generate_varlen_mask_params(cu)
    out = {"starts": s, "ends": e}
    qpos = torch.tensor([11, 0, 4, 3, 8])
    out["for_positions"] = list(M.generate_varlen_mask_params_for_positions(cu, qpos))
    kpos = torch.randperm(12)
    out["valid_from_starts_ends"] = M.build_valid_mask_from_starts_ends(s, e, kpos)
    out["causal_from_positions"] = M.build_causal_mask_from_positions(qpos, kpos)
    scores = torch.randn(2, 3, 12, 12)
    out["scores_masked"] = M.apply_starts_ends_mask_to_scores(scores, s, e, kpos)
    idx = torch.randint(0, 12, (2, 5, 4))
    ok = torch.rand(2, 5, 4) > 0.3
    sc = torch.randn(2, 5, 4)
    out["sorted_topk"] = list(M.sort_topk_by_index(idx, ok, sk=12, topk_scores=sc))
    logits = torch.randn(3, 6, 9)
    valid = torch.rand(3, 6, 9) > 0.4
    valid[1, 2] = False                                                 # fully masked row
    out["masked_softmax"] = M.masked_softmax(logits, valid)
    out["masked_log_softmax"] = M.masked_log_softmax(logits, valid)
    out["masked_softmax_inplace"] = M.masked_softmax_inplace(logits.clone(), valid)
    out["additive_mask"] = [list(M.prepare_additive_mask(m, sq=6, sk=9, b=3, device=device))
                            for m in (None, torch.randn(6, 9).masked_fill(torch.rand(6, 9) > 0.5, float("-inf")))]
    out["sparse_validity"] = M.apply_sparse_validity_to_index_mask(torch.zeros(1, 12, 12), row_mask=None, varlen_starts=s, varlen_ends=e, key_positions=None)
    return out


def test_masking_helpers_match_reference():
    from megatron_b200.core.transformer.experimental_attention_variant import dsa_masking as M

    want = _golden("dsa_masking")
    got = _masking_outputs(M, "cpu")
    assert sorted(got) == sorted(want)
    for k in ("starts", "ends", "valid_from_starts_ends", "causal_from_positions", "scores_masked", "sparse_validity"):
        assert torch.equal(got[k], want[k]), k
    for k in ("for_positions", "sorted_topk"):
        assert len(got[k]) == len(want[k]) and all(torch.equal(a, b) for a, b in zip(got[k], want[k])), k
    for gm, wm in zip(got["additive_mask"], want["additive_mask"], strict=True):
        assert len(gm) == len(wm) and all(torch.equal(a, b) for a, b in zip(gm, wm))
    assert torch.allclose(got["masked_softmax"], want["masked_softmax"], atol=1e-7)
    assert torch.allclose(got["masked_log_softmax"], want["masked_log_softmax"], atol=1e-6)
    assert torch.allclose(got["masked_softmax_inplace"], want["masked_softmax_inplace"], atol=1e-7)
    assert not torch.isnan(got["masked_softmax"]).any() and got["masked_softmax"][1, 2].abs().sum() == 0
    s, e = got["starts"], got["ends"]
    with pytest.raises(ValueError):
        M.normalize_varlen_bounds(mask=torch.zeros(2, 2), varlen_starts=s, varlen_ends=e, key_positions=None, sk=12, device="cpu")


def test_valid_rows_from_padded_packing():
    from types import SimpleNamespace

    from megatron_b200.core.transformer.experimental_attention_variant.dsa_masking import extract_query_valid_rows_from_packed_seq_params, normalize_query_valid_rows

    p = SimpleNamespace(cu_seqlens_q=torch.tensor([0, 3, 5]), cu_seqlens_q_padded=torch.tensor([0, 4, 8]))
    v = extract_query_valid_rows_from_packed_seq_params(p, 8, "cpu")
    assert v.tolist() == [True, True, True, False, True, True, False, False]
    assert normalize_query_valid_rows(v, b=2, sq=8, device="cpu").shape == (2, 8)


def _routing_scores_outputs(M):
    torch.manual_seed(0)
    logits = torch.randn(10, 8)
    pad = torch.rand(10) > 0.7
    out = {}
    for fn in ("softmax", "sigmoid", "sqrtsoftplus"):
        for pm_name, pm in (("nopad", None), ("pad", pad)):
            out[f"{fn}_{pm_name}"] = list(M.compute_routing_scores_for_aux_loss(logits, 2, fn, padding_mask=pm))
    return out


def test_moe_utils_additions_match_reference():
    from megatron_b200.core.transformer.moe import moe_utils as M

    want = _golden("moe_routing_scores")
    got = _routing_scores_outputs(M)
    assert sorted(got) == sorted(want)
    for k, (m1, s1) in got.items():
        m2, s2 = want[k]
        assert torch.equal(m1.bool(), m2.bool()) and torch.allclose(s1, s2, atol=1e-7), k
    cnt = torch.tensor([[5.0, 1.0, 3.0, 3.0], [2.0, 2.0, 2.0, 2.0]])
    new = M.get_updated_expert_bias(cnt.clone(), torch.zeros(2, 4), 0.01)
    assert torch.allclose(new, torch.tensor([[-0.01, 0.01, 0.0, 0.0], [0.0, 0.0, 0.0, 0.0]]))
    rm = torch.tensor([[1, 1, 0], [0, 0, 0], [1, 0, 1]], dtype=torch.bool)
    g, loc, tot = M.get_tokens_per_expert_and_token_count(rm, None, topk=2, with_padding_mask=True)
    assert g.tolist() == [2, 1, 1] and float(loc) == 2.0 and float(tot) == 2.0
    # fp32 gating of bf16 activations: gradients return in bf16 and match autograd of the plain formula
    x = torch.randn(6, 16, dtype=torch.bfloat16, requires_grad=True)
    w = torch.randn(4, 16, dtype=torch.bfloat16, requires_grad=True)
    out = M.router_gating_linear(x, w, None, torch.float32)
    assert out.dtype == torch.float32
    gout = torch.randn_like(out)
    gx, gw = torch.autograd.grad(out, (x, w), gout)
    rx, rw = torch.autograd.grad(x.float() @ w.float().t(), (x, w), gout)
    assert gx.dtype == torch.bfloat16 and torch.allclose(gx.float(), rx.float(), atol=2e-2, rtol=2e-2) and torch.allclose(gw.float(), rw.float(), atol=5e-2, rtol=2e-2)

    class C:
        fp8, fp4, fp8_recipe = "e4m3", None, "mxfp8"
    assert M.get_align_size_for_quantization(C) == 128


HYBRID_PATTERN = "M-M-|M-M*-/MM/MM"


def _hybrid_outputs(M):
    ratios = {(n, ar, mr): M.pattern_from_ratios(n, ar, mr)
              for n in (1, 7, 24, 52, 56) for ar, mr in ((0.0, 0.0), (0.1, 0.0), (0.08, 0.5), (0.25, 0.25), (0.5, 0.5), (1.0, 0.0))}
    p = M.parse_hybrid_pattern(HYBRID_PATTERN)
    return {"pattern_from_ratios": [[list(k), v] for k, v in ratios.items()],
            "parsed": [p.main_pattern, p.mtp_pattern, p.mtp_num_depths],
            "total_layers": M.get_hybrid_total_layer_count(HYBRID_PATTERN),
            "segments": M.get_hybrid_total_pipeline_segment_count(HYBRID_PATTERN),
            "layer_counts": dict(M.get_hybrid_layer_counts(HYBRID_PATTERN)),
            "layer_maps": {k: dict(v) for k, v in M.get_layer_maps_from_layer_type_list(list("M*M-*")).items()}}


def test_hybrid_pattern_helpers_match_reference():
    from megatron_b200.core.models.hybrid import hybrid_layer_allocation as M

    want = _golden("hybrid_layer_allocation")
    got = _hybrid_outputs(M)
    assert got["pattern_from_ratios"] == want["pattern_from_ratios"]
    assert got["parsed"] == want["parsed"]
    assert got["total_layers"] == want["total_layers"] == 9
    assert got["segments"] == want["segments"] == 2
    assert all(got["layer_counts"][k] == v for k, v in want["layer_counts"].items())
    assert M.select_pipeline_segment("M-M-|M-M*-", pp_rank=1, pp_size=2) == (list("M-M*-"), 4)
    assert M.select_pipeline_segment("MM|**|--|EE", pp_rank=1, pp_size=2, vp_stage=1) == (list("EE"), 6)
    assert M.select_pipeline_segment("MMMMMMMM", pp_rank=2, pp_size=4) == (list("MM"), 4)
    assert M.select_pipeline_segment("M" * 10, pp_rank=3, pp_size=4, first_stage_layers=1, last_stage_layers=3) == (list("MMM"), 7)
    with pytest.raises(ValueError):
        M.select_pipeline_segment("MMM", pp_rank=0, pp_size=2)
    with pytest.raises(ValueError):
        M.parse_hybrid_pattern("MM/M*/MM")
    assert all(got["layer_maps"][k] == v for k, v in want["layer_maps"].items())
