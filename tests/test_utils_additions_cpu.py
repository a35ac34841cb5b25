"""Round-2 helpers in core/utils.py and core/transformer/utils.py."""
import asyncio
import warnings

import pytest
import torch

from dist_utils import run_distributed


def test_small_helpers():
    from megatron_b200.core import config as mcfg, utils as U

    assert U.null_decorator(len) is len and U.null_decorator(nopython=True)(len) is len
    assert U.round_up_to_nearest_multiple(13, 8) == 16 and U.round_up_to_nearest_multiple(16, 8) == 16
    assert U.accepts_parameter(lambda a, b=1: 0, "b") and not U.accepts_parameter(lambda a: 0, "b") and U.accepts_parameter(lambda **k: 0, "zz")
    box = U.WrappedTensor(torch.ones(2))
    assert box.unwrap().sum() == 2
    with pytest.raises(RuntimeError):
        box.unwrap()
    assert U.get_torch_version().major >= 2 and not U.is_mamba_min_version("0.0.1")
    lin = torch.nn.Linear(2, 2)
    seq = torch.nn.Sequential(lin)
    assert U.is_submodule(lin, seq) and not U.is_submodule(seq, seq) and U.is_submodule(seq, seq, strict=False)

    @U.experimental_api
    def f():
        return 1

    @U.experimental_cls("0.20")
    class C:
        def __init__(self):
            self.x = 1
    mcfg.set_experimental_flag(False)
    with pytest.raises(U.ExperimentalNotEnabledError):
        f()
    with pytest.raises(U.ExperimentalNotEnabledError):
        C()
    mcfg.set_experimental_flag(True)
    assert f() == 1 and C().x == 1
    mcfg.set_experimental_flag(False)

    @U.deprecate_args("old")
    def g(a, new=0):
        return a + new
    with warnings.catch_warnings(record=True) as w:
        warnings.simplefilter("always")
        assert g(1, old=5, new=2) == 3 and any("old" in str(x.message) for x in w)
    assert U.deprecate_inference_params("ctx", "params") == "ctx"

    @U.trace_async_exceptions
    async def boom():
        raise ValueError("x")
    with pytest.raises(ValueError):
        U.get_asyncio_loop().run_until_complete(boom())
    std = torch.stack([U.mup_scaled_init_method_normal(0.02, 4, 4.0)(torch.empty(4096)).std() for _ in range(4)]).mean()
    assert abs(float(std) - 0.02 / (8 ** 0.5) / 2) < 2e-4


def test_flatten_batch_for_packed_sequences():
    from megatron_b200.core.utils import flatten_batch_for_packed_sequences

    batch = {"tokens": torch.arange(16).view(2, 8), "labels": torch.arange(16).view(2, 8), "loss_mask": torch.ones(2, 8), "position_ids": torch.arange(8).repeat(2, 1),
             "cu_seqlens": torch.tensor([[0, 3, 8, 8], [0, 5, 6, 8]]), "max_seqlen": torch.tensor([5, 5])}
    out = flatten_batch_for_packed_sequences(batch)
    assert out["tokens"].shape == (1, 16) and out["cu_seqlens"].tolist() == [[0, 3, 8, 13, 14, 16]] and out["max_seqlen"].tolist() == [5]


def _tp_batch_worker(rank, world):
    import torch.distributed as dist

    from megatron_b200.core.utils import get_batch_on_this_tp_rank

    full = {"tokens": torch.arange(12).view(2, 6), "labels": torch.arange(12).view(2, 6) + 1, "loss_mask": torch.rand(2, 6), "position_ids": torch.arange(6).repeat(2, 1),
            "attention_mask": None, "cu_seqlens": torch.tensor([[0, 2, 6]], dtype=torch.int32), "max_seqlen": torch.tensor([4], dtype=torch.int32)}
    torch.manual_seed(0)
    full["loss_mask"] = torch.rand(2, 6)
    mine = full if rank == 0 else None
    out = get_batch_on_this_tp_rank(mine, has_cu_seqlens=True, broadcast_src_rank=0, broadcast_group=dist.group.WORLD, tp_rank=rank)
    for k in ("tokens", "labels", "loss_mask", "position_ids", "cu_seqlens", "max_seqlen"):
        assert torch.equal(out[k], full[k]) and out[k].dtype == full[k].dtype, k
    assert out["attention_mask"] is None
    # last pipeline stage without MTP: no tokens travel
    out = get_batch_on_this_tp_rank(mine, broadcast_src_rank=0, broadcast_group=dist.group.WORLD, tp_rank=rank, pipeline_model_parallel_size=2,
                                    is_pipeline_first_stage=False, is_pipeline_last_stage=True)
    if rank != 0:
        assert out["tokens"] is None and torch.equal(out["labels"], full["labels"])
    return True


def test_get_batch_on_this_tp_rank_two_broadcasts():
    assert all(run_distributed(_tp_batch_worker, 2))


def test_transformer_utils_additions():
    from megatron_b200.core.transformer import utils as TU

    m = TU.get_sliding_window_causal_mask(4, 6, (2, 0))
    # query 0 sits at key position 2: sees keys 0..2
    assert m[0].tolist() == [False, False, False, True, True, True] and m[3].tolist() == [True, True, True, False, False, False]
    assert TU.is_layer_window_attention((128, 0), 4, 3) and not TU.is_layer_window_attention((128, 0), 4, 4) and not TU.is_layer_window_attention(None, None, 1)
    assert TU.is_layer_window_attention((128, 0), [1, 0, 1], 3) and not TU.is_layer_window_attention((128, 0), [1, 0, 1], 2)
    x = torch.randn(64)
    assert torch.allclose(TU.openai_gelu(x), torch.nn.functional.gelu(x, approximate="tanh"), atol=1e-6)
    assert torch.allclose(TU.erf_gelu(x), torch.nn.functional.gelu(x), atol=1e-6)
    assert torch.equal(TU.cat_with_oom_fallback([torch.ones(2), torch.zeros(1)]), torch.tensor([1.0, 1.0, 0.0]))

    class Cfg:
        sequence_parallel = True
        cuda_graph_impl = "local"

    class Layer(torch.nn.Module):
        def __init__(self, cfg):
            super().__init__()
            self.config, self.sequence_parallel = cfg, True
            self.w = torch.nn.Parameter(torch.zeros(1))
            self.w.sequence_parallel = True

    cfg = Cfg()
    net = torch.nn.Sequential(Layer(cfg), Layer(cfg))
    TU.set_model_to_sequence_parallel(net, False, exclude_modules=["1"])
    assert net[0].sequence_parallel is False and net[0].w.sequence_parallel is False and net[1].sequence_parallel is True and cfg.sequence_parallel is False
    assert TU.set_model_config_attribute(net, "cuda_graph_impl", "none") == 1 and cfg.cuda_graph_impl == "none"
    TU.toggle_cuda_graphs(net, "full")
    assert cfg.cuda_graph_impl == "full"


# a small fixed checkpoint directory whose integrity manifest the unmodified reference wrote into tests/golden/reference/integrity.json
INTEGRITY_FILES = {"__0_0.distcp": bytes(range(256)) * 5, "common.pt": b"common state", "metadata.json": b'{"sharded_backend": "torch_dist"}'}


def test_checkpoint_integrity_manifest_and_strict_helpers(tmp_path):
    import json
    import os
    import shutil

    from megatron_b200.core import dist_checkpointing as dc
    from megatron_b200.core.dist_checkpointing import validation as V
    from megatron_b200.core.dist_checkpointing.core import CheckpointingException
    from megatron_b200.core.dist_checkpointing.mapping import ShardedTensor

    ck = str(tmp_path / "ck")
    os.makedirs(ck)
    sd = {"a": ShardedTensor.from_rank_offsets("a", torch.arange(6.0)), "b": ShardedTensor.from_rank_offsets("b", torch.ones(3))}
    dc.save(sd, ck)
    V.verify_checkpoint(ck)
    with pytest.raises(CheckpointingException):
        V.verify_checkpoint(str(tmp_path / "nope"))
    V.save_integrity_manifest(ck)
    V.verify_integrity_manifest(ck)
    # the unmodified reference writes the same manifest for the same files (tests/golden/reference/integrity.json), and ours accepts the reference's
    fixed = tmp_path / "fixed"
    fixed.mkdir()
    for name, data in INTEGRITY_FILES.items():
        (fixed / name).write_bytes(data)
    V.save_integrity_manifest(str(fixed))
    golden = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference", "integrity.json")
    with open(golden) as f, open(fixed / "integrity.json") as g:
        assert json.load(g) == json.load(f)
    shutil.copyfile(golden, fixed / "integrity.json")
    V.verify_integrity_manifest(str(fixed))
    victim = next(n for n in sorted(os.listdir(ck)) if n.endswith(".distcp"))
    with open(os.path.join(ck, victim), "r+b") as f:
        f.seek(10)
        f.write(b"\xff\xfe")
    with pytest.raises(CheckpointingException, match="hash mismatch"):
        V.verify_integrity_manifest(ck)
    assert V.parse_strict_flag("log_all") is V.StrictHandling.LOG_ALL and V.parse_strict_flag(V.StrictHandling.RAISE_ALL) is V.StrictHandling.RAISE_ALL
    with pytest.raises(ValueError):
        V.parse_strict_flag("bogus")
    pruned = V.adjust_non_strict_load({"m": dict(sd), "l": [sd["a"]]}, {"a"})
    assert list(pruned["m"]) == ["b"] and pruned["l"] == []
    with pytest.raises(CheckpointingException):
        V.maybe_report_missing_and_unexpected_keys(V.StrictHandling.RAISE_ALL, {"x"}, set())
    V.maybe_report_missing_and_unexpected_keys(V.StrictHandling.LOG_ALL, {"x"}, {"y"})
    V.maybe_report_missing_and_unexpected_keys(V.StrictHandling.RAISE_UNEXPECTED, {"x"}, set())     # only "unexpected" raises here


def test_full_iteration_graph_static_buffers_on_cpu():
    from megatron_b200.core.full_cuda_graph import FullCudaGraphWrapper, StaticBufferLoader, clone_tensors_in_struct, copy_tensors_in_struct

    a = {"tokens": torch.arange(6).view(2, 3), "meta": ("x", [torch.ones(2)])}
    s = clone_tensors_in_struct(a, "cpu")
    ptr = s["tokens"].data_ptr()
    b = {"tokens": torch.arange(6).view(2, 3) + 10, "meta": ("y", [torch.zeros(2)])}
    s = copy_tensors_in_struct(s, b)
    assert s["tokens"].data_ptr() == ptr and s["tokens"][0, 0] == 10 and s["meta"][0] == "y" and s["meta"][1][0].sum() == 0
    with pytest.raises(ValueError):
        copy_tensors_in_struct(s, {"tokens": torch.zeros(2, 4), "meta": b["meta"]})
    seen = []

    def fwd_bwd(*, data_iterator, num_microbatches, forward_only=False):
        out = [next(data_iterator) for _ in range(num_microbatches)]
        seen.append([(o["x"].data_ptr(), int(o["x"].sum())) for o in out])
        return [o["x"].sum() for o in out]

    w = FullCudaGraphWrapper(fwd_bwd, cuda_graph_warmup_steps=1, device="cpu")
    data = iter([{"x": torch.full((2,), float(i))} for i in range(8)])
    w(data_iterator=data, num_microbatches=2)
    w(data_iterator=data, num_microbatches=2)
    w(data_iterator=data, num_microbatches=2, forward_only=True)
    assert [p for p, _ in seen[0]] == [p for p, _ in seen[1]], "the same static buffers are read every step"
    assert [v for _, v in seen[0]] == [0, 2] and [v for _, v in seen[1]] == [4, 6] and [v for _, v in seen[2]] == [8, 10]
    assert {p for p, _ in seen[2]}.isdisjoint({p for p, _ in seen[0]}), "validation has its own buffers"
    ld = StaticBufferLoader("cpu")
    with pytest.raises(IndexError):
        ld.load("training", 1, {"x": torch.zeros(1)})


def _fault_plan_worker(rank, world):
    import time
    from types import SimpleNamespace

    from megatron_b200.core import fault_injector as F

    cfg = SimpleNamespace(fault_injector_ranks=None, fault_injector_num_ranks=1, fault_injector_fault_types="workload_exc", fault_injector_fault_probabilities=None,
                          fault_injector_fault_delay=0.05, fault_injector_delay_start_iteration=None, fault_injector_mtti_seconds=None,
                          fault_injector_offset_seconds=None, fault_injector_seed=7 + rank)          # different seeds: only rank 0's draw counts
    assert F.should_setup_fault_injection_at_start(cfg) and not F.should_setup_fault_injection_at_iteration(cfg, 3)
    inj = F.setup_fault_injection(cfg)
    time.sleep(0.3)
    hit = False
    if inj is not None:
        try:
            inj.maybe_raise()
        except F.InjectedFaultError:
            hit = True
    return (inj is not None, hit)


def test_fault_plan_is_drawn_on_rank0_and_broadcast():
    from types import SimpleNamespace

    from megatron_b200.core import fault_injector as F

    out = run_distributed(_fault_plan_worker, 3)
    armed = [o[0] for o in out]
    assert armed[0] is False and sum(armed) == 1, "one random rank, never rank 0"
    assert all(hit == a for a, hit in out)
    cfg = SimpleNamespace(fault_injector_ranks="1,2", fault_injector_num_ranks=None, fault_injector_fault_delay=None, fault_injector_mtti_seconds=100.0,
                          fault_injector_offset_seconds=5.0, fault_injector_seed=1, fault_injector_fault_types="sigkill,gpu_sleep", fault_injector_fault_probabilities="0,1")
    assert F.get_fault_ranks(cfg, 4) == [1, 2] and F.get_fault(cfg) is F.Fault.GPU_SLEEP and F.get_fault_delay(cfg) > 5.0


def test_verify_integrity_through_save_and_load(tmp_path):
    import os

    from megatron_b200.core import dist_checkpointing as dc
    from megatron_b200.core.dist_checkpointing.core import CheckpointingException
    from megatron_b200.core.dist_checkpointing.mapping import ShardedTensor

    ck = str(tmp_path / "ck")
    os.makedirs(ck)
    dc.save({"a": ShardedTensor.from_rank_offsets("a", torch.arange(4.0))}, ck, verify_integrity=True)
    assert os.path.isfile(os.path.join(ck, "integrity.json"))
    out = dc.load({"a": ShardedTensor.from_rank_offsets("a", torch.zeros(4))}, ck, verify_integrity=True)
    assert torch.equal(out["a"], torch.arange(4.0))
    with open(os.path.join(ck, "common.pt"), "ab") as f:
        f.write(b"x")
    with pytest.raises(CheckpointingException, match="hash mismatch"):
        dc.load({"a": ShardedTensor.from_rank_offsets("a", torch.zeros(4))}, ck, verify_integrity=True)
