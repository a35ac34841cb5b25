"""Training-program support: masks, writers, one-logger, signal handler, fault-tolerance monitor, activation logging, determinism, SFT / FIM data."""
import json
import os
import signal
import time

import numpy as np
import pytest
import torch


def test_ltor_masks_reset_positions_and_attention():
    from megatron_b200.training.utils import get_ltor_masks_and_position_ids

    eod = 9
    data = torch.tensor([[1, 2, eod, 3, 4, 5, eod, 6], [1, 2, 3, 4, 5, 6, 7, 8]])
    att, loss, pos = get_ltor_masks_and_position_ids(data, eod, reset_position_ids=True, reset_attention_mask=True, eod_mask_loss=True)
    assert pos[0].tolist() == [0, 1, 2, 0, 1, 2, 3, 0] and pos[1].tolist() == list(range(8))
    assert loss[0].tolist() == [1, 1, 0, 1, 1, 1, 0, 1]
    # brute force: token i may attend token j iff j <= i and same document
    doc = [0, 0, 0, 1, 1, 1, 1, 2]
    for i in range(8):
        for j in range(8):
            assert bool(att[0, 0, i, j]) == (not (j <= i and doc[i] == doc[j]))
    assert torch.equal(att[1, 0], torch.ones(8, 8, dtype=torch.bool).triu(1))
    att2, _, pos2 = get_ltor_masks_and_position_ids(data, eod)
    assert att2.shape == (1, 1, 8, 8) and pos2[0].tolist() == list(range(8))


def test_scalar_writer_one_logger_and_wandb_hooks(tmp_path):
    from types import SimpleNamespace

    from megatron_b200.training import global_vars as gv
    from megatron_b200.training import wandb_utils

    args = SimpleNamespace(tensorboard_dir=str(tmp_path / "tb"), wandb_project="p", wandb_save_dir=str(tmp_path / "wb"), save=str(tmp_path), enable_one_logger=True,
                           timing_log_level=0, timing_log_option="minmax", world_size=1)
    os.environ["WANDB_MODE"] = "offline"
    gv.set_global_variables(args)
    try:
        tb = gv.get_tensorboard_writer()
        tb.add_scalar("lm loss", 2.5, 10)
        tb.flush()
        ol = gv.get_one_logger()
        ol.on_train_start(0, 0, 100, 8, 10, str(tmp_path), False, True, 0.0)
        ol.track_iteration(0.5, 4, 8, 1e12)
        ol.track_iteration(1.5, 4, 8, 1e12)
        ol.on_save_checkpoint_start(False)
        ol.on_save_checkpoint_end(2, False)
        ol.on_train_end()
        assert ol.store_get("train_iterations_time_msecs_avg") == 1000.0 and ol.store_get("train_samples_end") == 8
        assert ol.store_get("last_successful_save_checkpoint_iteration") == 2
        recs = [json.loads(l) for l in open(ol.path)]
        assert any("app_train_loop_finish_time" in r for r in recs)
        w = gv.get_wandb_writer()
        if not hasattr(w, "Artifact"):       # offline JSON sink
            ck = tmp_path / "iter_0000002"
            ck.mkdir()
            tracker = tmp_path / "latest_checkpointed_iteration.txt"
            tracker.write_text("2")
            wandb_utils.on_save_checkpoint_success(str(ck), str(tracker), str(tmp_path), 2)
            wandb_utils.on_load_checkpoint_success(str(ck), str(tmp_path))
            assert [r for r in w.read() if r["tag"].startswith("checkpoint/")]
    finally:
        gv.unset_global_variables()


def test_distributed_signal_handler_single_process():
    from megatron_b200.training.dist_signal_handler import DistributedSignalHandler

    prev = signal.getsignal(signal.SIGUSR1)
    with DistributedSignalHandler(signal.SIGUSR1) as h:
        assert h.signals_received() == [False]
        os.kill(os.getpid(), signal.SIGUSR1)
        time.sleep(0.05)
        assert h.any_received()
    assert signal.getsignal(signal.SIGUSR1) == prev


def test_fault_tolerance_monitor_learns_timeouts_and_detects_hang(tmp_path):
    from megatron_b200.training.ft_integration import FaultToleranceMonitor

    mon = FaultToleranceMonitor(rank=0, save_dir=str(tmp_path), timeouts={"step": 0.3}, min_samples=3, poll_interval=0.05, abort=False, safety_factor=4.0).start()
    for _ in range(3):
        mon.start_section("step")
        time.sleep(0.02)
        mon.end_section("step")
    assert mon.expired is None
    t = mon.calc_timeouts()
    assert 1.0 <= t["step"] < 2.0 and json.load(open(tmp_path / "ft_state.json"))["timeouts"]["step"] == t["step"]
    mon.timeouts["step"] = 0.2
    mon.start_section("step")
    time.sleep(0.6)                      # never ends: the watchdog must fire
    assert mon.expired is not None and mon.expired["section"] == "step"
    assert json.load(open(tmp_path / "hang_rank0.json"))["section"] == "step"
    mon.shutdown()
    # a restarted monitor starts from the learned values
    assert FaultToleranceMonitor(save_dir=str(tmp_path)).timeouts["step"] == t["step"]


def test_activation_and_dgrad_logging(tmp_path):
    from megatron_b200.training.activation_logging import ActivationLogger, DgradLogger, WgradLogger

    class Blk(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.self_attention = torch.nn.Linear(8, 8)
            self.mlp = torch.nn.Linear(8, 8)

        def forward(self, x):
            return self.mlp(torch.relu(self.self_attention(x)))

    m = torch.nn.Sequential(Blk(), Blk())
    act, dg, wg = (cls(m, str(tmp_path), interval=2, pattern=r".*(self_attention|mlp)$") for cls in (ActivationLogger, DgradLogger, WgradLogger))
    for it in (1, 2):
        armed = [l.begin_iteration(it) for l in (act, dg, wg)]
        assert armed == [it == 2] * 3
        x = torch.randn(4, 8, requires_grad=True)
        m(x).sum().backward()
        wg.collect() if armed[0] else None
        paths = [l.end_iteration() for l in (act, dg, wg)]
        assert all((p is not None) == (it == 2) for p in paths)
    a = json.load(open(paths[0]))
    d = json.load(open(paths[1]))
    w = json.load(open(paths[2]))
    assert set(a) == {"chunk0.0.self_attention", "chunk0.0.mlp", "chunk0.1.self_attention", "chunk0.1.mlp"} and set(d) == set(a)
    assert a["chunk0.1.mlp"]["shape"] == [4, 8] and abs(d["chunk0.1.mlp"]["norm"] - (32 ** 0.5)) < 1e-5 and "chunk0.0.mlp.weight" in w
    assert not act.handles and len(m[0].mlp._forward_hooks) == 0


def test_determinism_digest_and_check():
    from megatron_b200.training.determinism import check_determinism, model_digest, tensor_digest

    torch.manual_seed(0)
    a = torch.randn(16)
    assert tensor_digest([a]) == tensor_digest([a.clone()]) != tensor_digest([a + 1e-7])
    lin = torch.nn.Linear(4, 4)
    d0 = model_digest(lin)
    with torch.no_grad():
        lin.weight[0, 0] += 1e-6
    assert model_digest(lin) != d0

    def run():
        torch.manual_seed(3)
        return [torch.randn(8) @ torch.randn(8, 8)]

    assert len(set(check_determinism(run, 3))) == 1
    import pytest

    with pytest.raises(RuntimeError):
        check_determinism(lambda: [torch.randn(4)], 2)


class _Tok:
    """Whitespace tokenizer with a growing vocabulary."""

    def __init__(self):
        self.v = {}

    def tokenize(self, s):
        return [self.v.setdefault(w, len(self.v) + 10) for w in s.replace("\n", " \n ").split(" ") if w]


def test_sft_dataset_masks_and_packing():
    from megatron_b200.training.datasets import SFTDataset, SFTDatasetConfig, pack_conversations

    assert pack_conversations([5, 3, 3, 2, 6], 8) == [[4, 3], [0, 1], [2]]
    tok = _Tok()
    convs = [[{"role": "user", "content": "hi there"}, {"role": "assistant", "content": "hello you"}],
             [{"role": "system", "content": "be brief"}, {"role": "user", "content": "q"}, {"role": "assistant", "content": "a"}]]
    ds = SFTDataset(convs, tok, SFTDatasetConfig(sequence_length=40, pad_token_id=0, pack=True))
    assert len(ds) == 1
    it = ds[0]
    assert it["tokens"].shape == (40,) and it["cu_seqlens"][0] == 0 and it["cu_seqlens"][-1] == 40
    n_docs = 2
    bounds = it["cu_seqlens"][: n_docs + 1].tolist()
    inv = {v: k for k, v in tok.v.items()}
    trained = [inv[int(t)] for t, m in zip(it["labels"], it["loss_mask"]) if m > 0]
    assert sorted(trained) == sorted(["hello", "you<|end|>", "\n", "a<|end|>", "\n"])     # assistant bodies (+ end-of-turn), nothing else
    for lo, hi in zip(bounds[:-1], bounds[1:]):
        assert it["position_ids"][lo:hi].tolist() == list(range(hi - lo))
        assert torch.equal(it["tokens"][lo + 1 : hi], it["labels"][lo : hi - 1].where(it["loss_mask"][lo : hi - 1] > 0, it["tokens"][lo + 1 : hi]))
    assert (it["labels"][it["loss_mask"] == 0] == -100).all()


def test_fim_transform_preserves_tokens_and_length():
    from megatron_b200.training.datasets import FIMConfig, GPTFIMDataset, apply_fim

    cfg = FIMConfig(fim_rate=1.0, fim_spm_rate=0.0, prefix_id=100, middle_id=101, suffix_id=102, pad_id=103, eod_id=104)
    doc = np.arange(10, 30)
    toks = np.concatenate([doc, [104], np.arange(40, 52)])
    out = apply_fim(toks, np.random.RandomState(0), cfg)
    assert len(out) == len(toks) and out[20] == 104
    first = out[:20]
    assert first[0] == 100 and 101 in first and 102 in first
    # PSM: prefix + middle + (suffix without its last three tokens) reassemble the document
    i_s, i_m = int(np.where(first == 102)[0][0]), int(np.where(first == 101)[0][0])
    p, s, m = first[1:i_s], first[i_s + 1 : i_m], first[i_m + 1 :]
    assert np.array_equal(np.concatenate([p, m, s]), doc[:17])
    spm = apply_fim(doc, np.random.RandomState(1), FIMConfig(fim_rate=1.0, fim_spm_rate=1.0, prefix_id=100, middle_id=101, suffix_id=102, eod_id=104))
    assert spm[0] == 100 and spm[1] == 102
    assert np.array_equal(apply_fim(doc, np.random.RandomState(0), FIMConfig(fim_rate=0.0, eod_id=104)), doc)

    class Base(torch.utils.data.Dataset):
        def __len__(self):
            return 4

        def __getitem__(self, i):
            t = torch.arange(10, 31) + i
            return {"tokens": t[:-1], "labels": t[1:], "loss_mask": torch.ones(20)}

    ds = GPTFIMDataset(Base(), cfg, seed=7)
    a, b = ds[2], ds[2]
    assert torch.equal(a["tokens"], b["tokens"]) and a["tokens"].shape == (20,) and torch.equal(a["tokens"][1:], a["labels"][:-1])


def _run_pretrain(tmp_path, extra, iters):
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, os.path.join(root, "pretrain_gpt.py"), "--num-layers", "2", "--hidden-size", "64", "--num-attention-heads", "4", "--ffn-hidden-size", "128",
           "--seq-length", "32", "--max-position-embeddings", "32", "--micro-batch-size", "2", "--global-batch-size", "4", "--train-iters", str(iters), "--lr", "1e-3",
           "--mock-data", "--tokenizer-type", "NullTokenizer", "--vocab-size", "127", "--log-interval", "2", "--distributed-backend", "gloo", "--swiglu",
           "--normalization", "RMSNorm", "--disable-bias-linear", "--position-embedding-type", "rope", "--untie-embeddings-and-output-weights",
           "--save", str(tmp_path / "ckpt"), "--load", str(tmp_path / "ckpt"), "--save-interval", "4", "--eval-iters", "0", "--lr-decay-iters", "100"] + extra
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", MASTER_PORT="29631", RANK="0", WORLD_SIZE="1", LOCAL_RANK="0", CUDA_VISIBLE_DEVICES="", WANDB_MODE="offline")
    r = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    return r.stdout


def test_pretrain_cli_writers_ft_activation_logs_and_resume(tmp_path):
    out = _run_pretrain(tmp_path, ["--tensorboard-dir", str(tmp_path / "tb"), "--enable-one-logger", "--enable-ft-package", "--log-activations-interval", "2",
                                   "--log-wgrad-interval", "4", "--activation-log-dir", str(tmp_path / "act"), "--exit-interval", "4"], iters=6)
    assert "iteration        4/" in out and "lm loss" in out and "iteration        6/" not in out
    tb_dir = tmp_path / "tb"
    assert tb_dir.exists() and any(tb_dir.iterdir())
    if (tb_dir / "scalars.jsonl").exists():
        tags = {json.loads(l)["tag"] for l in open(tb_dir / "scalars.jsonl")}
        assert {"lm loss", "iteration-time", "learning-rate"} <= tags
    acts = sorted(os.listdir(tmp_path / "act"))
    assert [a for a in acts if a.startswith("activation_iter0000002")] and [a for a in acts if a.startswith("wgrad_iter0000004")]
    assert json.load(open(tmp_path / "ckpt" / "ft_state.json"))["timeouts"]["checkpointing"] >= 1.0 if (tmp_path / "ckpt" / "ft_state.json").exists() else True
    recs = [json.loads(l) for l in open(tmp_path / "ckpt" / "one_logger.jsonl")]
    assert any(r.get("tracked_train_iterations") == 4 for r in recs)
    # resume: picks up at iteration 4 and continues to 6
    out2 = _run_pretrain(tmp_path, [], iters=6)
    assert "iteration        6/" in out2 and "iteration        2/" not in out2


def test_pretrain_cli_non_persistent_checkpoints_and_load_policy(tmp_path):
    """--non-persistent-ckpt-type global: a recovery checkpoint every 2 iterations beside the persistent series (every 4, cached save plans); the restart resumes
    from the NEWEST of the two (iteration 6, non-persistent), then a fresh run elsewhere starts from it as --pretrained-checkpoint weights at iteration 0."""
    common = ["--non-persistent-save-interval", "2", "--non-persistent-ckpt-type", "global", "--ckpt-assume-constant-structure", "--ckpt-fully-parallel-load",
              "--dist-ckpt-strictness", "log_all", "--log-progress"]
    out = _run_pretrain(tmp_path, common + ["--exit-interval", "6"], iters=8)
    prog = (tmp_path / "ckpt" / "progress.txt").read_text().splitlines()
    assert prog[0].split("\t")[3] == "Starting job" and any("Saved checkpoint\titeration: 4" in l for l in prog) and "FLOPs so far" in prog[-1]
    assert "iteration        6/" in out and "iteration        8/" not in out
    np_dir = tmp_path / "ckpt" / "non_persistent"
    assert (np_dir / "latest_checkpointed_iteration.txt").read_text().strip() == "6"
    assert sorted(d for d in os.listdir(np_dir) if d.startswith("iter_")) == ["iter_0000006"]                   # only the newest is kept
    # exit at 6 also wrote the persistent series' iteration 6; remove it so that the non-persistent one is strictly newer
    import shutil

    shutil.rmtree(tmp_path / "ckpt" / "iter_0000006")
    (tmp_path / "ckpt" / "latest_checkpointed_iteration.txt").write_text("4")
    out2 = _run_pretrain(tmp_path, common, iters=8)
    assert "loaded non_persistent_global checkpoint" in out2 and "at iteration 6" in out2 and "iteration        8/" in out2 and "iteration        6/" not in out2
    # finetune-style start from pretrained weights: nothing in --load, iteration restarts at 0
    ft = tmp_path / "ft"
    out3 = _run_pretrain(ft, ["--pretrained-checkpoint", str(tmp_path / "ckpt"), "--exit-interval", "2"], iters=4)
    assert "loaded pretrained checkpoint" in out3 and "iteration        2/" in out3
    # --exit-on-missing-checkpoint
    out4 = _run_pretrain(tmp_path / "none", ["--exit-on-missing-checkpoint"], iters=2)
    assert "no checkpoint found" in out4 and "iteration        2/" not in out4


def _run_pretrain_world(tmp_path, extra, iters, world, port):
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr", "127.0.0.1", "--master-port", str(port),
           os.path.join(root, "pretrain_gpt.py"), "--num-layers", "2", "--hidden-size", "64", "--num-attention-heads", "4", "--ffn-hidden-size", "128",
           "--seq-length", "32", "--max-position-embeddings", "32", "--micro-batch-size", "2", "--global-batch-size", "8", "--train-iters", str(iters), "--lr", "1e-3",
           "--mock-data", "--tokenizer-type", "NullTokenizer", "--vocab-size", "127", "--log-interval", "1", "--distributed-backend", "gloo", "--swiglu",
           "--normalization", "RMSNorm", "--disable-bias-linear", "--position-embedding-type", "rope", "--untie-embeddings-and-output-weights", "--seed", "11",
           "--save", str(tmp_path / "ckpt"), "--load", str(tmp_path / "ckpt"), "--save-interval", "100", "--eval-iters", "0", "--lr-decay-iters", "100"] + extra
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="", WANDB_MODE="offline")
    r = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    return r.stdout


def _losses(out):
    import re

    return [float(x) for x in re.findall(r"lm loss: ([0-9.E+-]+)", out)]


def test_pretrain_cli_megatron_fsdp_matches_ddp(tmp_path):
    """--use-megatron-fsdp (ZeRO-3 units + FSDPOptimizer on the master shards) on 2 gloo ranks follows the same loss curve as plain DDP + Adam, saves, and resumes."""
    ddp = _losses(_run_pretrain_world(tmp_path / "ddp", ["--exit-interval", "4"], 4, 2, 29641))
    fs_out = _run_pretrain_world(tmp_path / "fsdp", ["--use-megatron-fsdp", "--data-parallel-sharding-strategy", "optim_grads_params", "--exit-interval", "4"], 6, 2, 29642)
    fs = _losses(fs_out)
    assert len(ddp) == 4 and len(fs) == 4
    assert all(abs(a - b) < 2e-3 * abs(a) for a, b in zip(ddp, fs)), (ddp, fs)
    assert fs[-1] < fs[0]
    out2 = _run_pretrain_world(tmp_path / "fsdp", ["--use-megatron-fsdp", "--data-parallel-sharding-strategy", "optim_grads_params"], 6, 2, 29643)
    assert "at iteration 4" in out2 and "iteration        6/" in out2 and "iteration        3/" not in out2
    assert _losses(out2)[0] < fs[0]                               # continues from the trained state, not from scratch


def test_config_logger_initialize_helpers_and_param_norm(tmp_path):
    from types import SimpleNamespace

    from megatron_b200.core.config_logger import has_config_logger_enabled, log_config_to_disk
    from megatron_b200.training import async_utils
    from megatron_b200.training.initialize import init_autoresume, set_random_seed
    from megatron_b200.training.utils import calc_params_l2_norm, report_memory

    cfg = SimpleNamespace(config_logger_dir=str(tmp_path / "cfg"))
    assert has_config_logger_enabled(cfg) and not has_config_logger_enabled(SimpleNamespace())
    lin = torch.nn.Linear(4, 4)
    f0 = log_config_to_disk(cfg, {"self": lin, "config": cfg, "dtype": torch.bfloat16, "fn": torch.relu, "module": lin, "shape": (2, 3)}, prefix="Linear", rank_str="0")
    f1 = log_config_to_disk(cfg, {"x": torch.zeros(2, 2)}, prefix="Linear", rank_str="0")
    d0, d1 = json.load(open(f0)), json.load(open(f1))
    assert f0.endswith("Linear.rank_0.iter0.json") and f1.endswith("iter1.json") and "self" not in d0
    assert d0["dtype"] == "torch.bfloat16" and d0["module"]["module"] == "Linear" and d1["x"] == {"tensor": [2, 2], "dtype": "torch.float32"}
    s = set_random_seed(77)
    a = torch.rand(3)
    set_random_seed(77)
    assert s == 77 and torch.equal(a, torch.rand(3))
    import pytest

    with pytest.raises(ValueError):
        set_random_seed(0)
    lin = torch.nn.Linear(3, 2, bias=False)
    with torch.no_grad():
        lin.weight.fill_(2.0)
    for p in lin.parameters():
        p.tensor_model_parallel = True
    assert abs(calc_params_l2_norm(lin) - (6 * 4.0) ** 0.5) < 1e-6
    assert "no CUDA device" in report_memory("x") or "allocated" in report_memory("x")
    sentinel = tmp_path / "resume_now"
    os.environ["MEGATRON_B200_AUTORESUME_FILE"] = str(sentinel)
    try:
        ar = init_autoresume()
        assert not ar.termination_requested()
        sentinel.write_text("1")
        assert ar.termination_requested()
        ar.request_resume()
        assert not sentinel.exists()
    finally:
        del os.environ["MEGATRON_B200_AUTORESUME_FILE"]
    # async queue wrapper: schedule a request, finalise it, queue is empty again
    from megatron_b200.core.dist_checkpointing.strategies.async_utils import AsyncRequest

    done = []
    async_utils.schedule_async_save(AsyncRequest(lambda p: open(p, "w").write("x"), (str(tmp_path / "blob"),), [lambda: done.append(1)]))
    assert not async_utils.is_empty_async_queue()
    async_utils.maybe_finalize_async_save(blocking=True)
    assert async_utils.is_empty_async_queue() and done == [1] and (tmp_path / "blob").read_text() == "x"
    async_utils.reset_persistent_async_worker()


def test_telemetry_spans_and_metrics(tmp_path):
    from megatron_b200.core import telemetry

    assert telemetry.span("train.iteration").__enter__() is None          # disabled: shared no-op
    rec = telemetry.SpanRecorder(path=str(tmp_path / "spans.jsonl"), enabled_groups=["train"])
    telemetry.set_recorder(rec)
    try:
        with telemetry.span("train.loop"):
            for i in range(3):
                with telemetry.span("train.iteration", iteration=i):
                    with telemetry.span("layer.attention"):        # group not enabled: skipped
                        time.sleep(0.001)
        try:
            with telemetry.span("train.optimizer_step"):
                raise ValueError
        except ValueError:
            pass
    finally:
        telemetry.set_recorder(None)
    s = rec.summary()
    assert s["train.iteration"]["count"] == 3 and s["train.loop"]["count"] == 1 and "layer.attention" not in s
    rows = [json.loads(l) for l in open(tmp_path / "spans.jsonl")]
    assert [r["parent"] for r in rows if r["name"] == "train.iteration"] == ["train.loop"] * 3
    assert [r for r in rows if r["name"] == "train.optimizer_step"][0]["error"] == "ValueError"
    m = telemetry.TrainingMetrics()
    m.record_iteration(iteration_time_s=0.5, tokens=1000, flops=2e12, world=2, loss=3.0, lr=1e-4)
    assert m.values["train.tokens_per_second"] == 2000 and m.values["train.tflops_per_gpu"] == 2.0 and m.values["train.lm_loss"] == 3.0


def _reference_golden(name):
    """Values computed by the unmodified reference (``tests/helpers/make_reference_golden.py``)."""
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference", name)) as f:
        return json.load(f)


FLOPS_BASE = dict(num_layers=32, hidden_size=4096, ffn_hidden_size=14336, num_attention_heads=32, num_query_groups=8, kv_channels=128, vocab_size=128256, seq_length=8192)
_MLA = dict(q_lora_rank=1536, kv_lora_rank=512, qk_head_dim=128, qk_pos_emb_head_dim=64, v_head_dim=128)
_LIN = dict(linear_key_head_dim=128, linear_value_head_dim=128, linear_num_key_heads=16, linear_num_value_heads=32, linear_conv_kernel_dim=4)
_THD_LENS = [1000, 3000, 4192] * 2
# name: (keyword arguments of our model on top of FLOPS_BASE, overrides of the reference's argument namespace, batch size, extra keywords of the reference's call)
FLOPS_CASES = {
    "llama3_8b": (dict(batch_size=4), {}, 4, {}),
    "moe_shared_expert": (dict(seq_length=4096, vocab_size=32000, batch_size=8, num_moe_experts=8, moe_router_topk=2, moe_shared_expert_intermediate_size=2048),
                          dict(num_experts=8, moe_router_topk=2, seq_length=4096, padded_vocab_size=32000, moe_shared_expert_intermediate_size=2048), 8, {}),
    "interleaved_moe_mtp": (dict(batch_size=2, num_moe_experts=16, moe_router_topk=4, moe_layer_freq=[0, 1] * 16, moe_ffn_hidden_size=2048, mtp_num_layers=1),
                            dict(num_experts=16, moe_router_topk=4, moe_layer_freq=[0, 1] * 16, moe_ffn_hidden_size=2048, mtp_num_layers=1), 2, {}),
    "mla": (dict(num_query_groups=32, batch_size=2, multi_latent_attention=True, **_MLA), dict(multi_latent_attention=True, group_query_attention=False, num_query_groups=32, **_MLA), 2, {}),
    # THD: real tokens and sum of squared sub-sequence lengths
    "thd": (dict(batch_size=2, seq_lens=_THD_LENS), {}, 2, dict(seqlen_squared_sum_in_batch=sum(n * n for n in _THD_LENS), total_real_tokens_in_batch=sum(_THD_LENS))),
    # gated-delta-net linear attention every layer but each 4th
    "gated_delta_net": (dict(batch_size=2, linear_attention_freq=4), dict(experimental_attention_variant="gated_delta_net", linear_attention_freq=4, **_LIN), 2, {}),
}


def test_flops_model_matches_reference_accounting():
    """The analytic FLOP count equals the reference's ``num_floating_point_operations`` (values stored in ``tests/golden/reference/training.json``)."""
    from megatron_b200.training.flops import causal_pairs, num_floating_point_operations as ours

    want = _reference_golden("training.json")["flops"]
    assert sorted(want) == sorted(FLOPS_CASES)
    close = lambda a, b: abs(a - b) <= 1e-9 * abs(b)
    for name, (kw, _, _, _) in FLOPS_CASES.items():
        assert close(ours(**{**FLOPS_BASE, **kw}), want[name]), name
    base = FLOPS_BASE
    # sliding window (ours only): never more than full causal attention, equal when the window covers the sequence
    assert ours(**base, batch_size=1, window_size=(1024, 0)) < ours(**base, batch_size=1) == ours(**base, batch_size=1, window_size=(8192, 0))
    assert causal_pairs(10, 4) == 4 * 10 - 8


def test_generated_flags_and_yaml_config(tmp_path):
    """Every config-dataclass field is a flag; a YAML file sets the same things; the command line wins; typos are errors."""
    import pytest

    from megatron_b200.training.arguments import build_full_parser, core_transformer_config_from_args, parse_args
    from megatron_b200.training.argument_utils import args_to_yaml, dataclass_from_args
    from megatron_b200.core.optimizer import OptimizerConfig

    parser = build_full_parser()
    n_flags = sum(1 for a in parser._actions if a.option_strings)
    assert n_flags > 350, n_flags                      # 184 hand-written + ~200 generated ones
    base = ["--num-layers", "2", "--hidden-size", "64", "--num-attention-heads", "4", "--seq-length", "32", "--max-position-embeddings", "32", "--micro-batch-size", "1",
            "--global-batch-size", "1", "--vocab-size", "128"]
    # generated flags reach the config objects
    from megatron_b200.training.arguments import validate_args

    a = validate_args(parse_args(base + ["--moe-router-num-groups", "2", "--no-apply-rope-fusion", "--adam-beta2", "0.9", "--layernorm-zero-centered-gamma"]), world_size=1)
    cfg = core_transformer_config_from_args(a)
    assert cfg.layernorm_zero_centered_gamma is True and getattr(cfg, "moe_router_num_groups", None) == 2
    assert dataclass_from_args(OptimizerConfig, a).adam_beta2 == 0.9
    # YAML: nested sections, kebab or snake keys; explicit flags win; unknown keys raise
    y = tmp_path / "run.yaml"
    y.write_text("model:\n  num_layers: 4\n  hidden-size: 128\n  qk_layernorm: true\noptimizer:\n  lr: 0.001\n  adam_beta2: 0.8\n")
    b = parse_args(base[2:] + ["--num-layers", "6", "--yaml-cfg", str(y)])
    assert b.num_layers == 6 and b.hidden_size == 64 and b.qk_layernorm is True and b.lr == 0.001 and b.adam_beta2 == 0.8
    c = parse_args(["--num-attention-heads", "4", "--seq-length", "32", "--max-position-embeddings", "32", "--micro-batch-size", "1", "--global-batch-size", "1",
                    "--vocab-size", "128", "--yaml-cfg", str(y)])
    assert c.num_layers == 4 and c.hidden_size == 128
    (tmp_path / "bad.yaml").write_text("num_layerz: 3\n")
    with pytest.raises(ValueError, match="num_layerz"):
        parse_args(base + ["--yaml-cfg", str(tmp_path / "bad.yaml")])
    assert "TransformerConfig" in args_to_yaml(b, (type(cfg),)) and "num_layers: 6" in args_to_yaml(b, (type(cfg),))


def test_reference_flag_table(monkeypatch):
    import pytest

    """Every flag of the reference's training parsers parses here; WIRED names are really consumed somewhere; inert ones are reported (and fatal under --strict)."""
    import glob
    import re

    from megatron_b200.training import reference_flags as rf
    from megatron_b200.training.arguments import build_full_parser, core_transformer_config_from_args, ddp_config_from_args, parse_args, validate_args
    from megatron_b200.training.reference_flags_table import REFERENCE_FLAG_TABLE

    parser = build_full_parser()
    known = {s for a in parser._actions for s in a.option_strings}
    assert len(REFERENCE_FLAG_TABLE) > 300 and all(f in known for row in REFERENCE_FLAG_TABLE for f in row[0])
    assert len(known) > 800
    # WIRED / ALWAYS_ON are honest: each dest is read by name outside the table module itself, or translated in reference_flags.py
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    src = ""
    for f in glob.glob(os.path.join(root, "megatron_b200/**/*.py"), recursive=True) + glob.glob(os.path.join(root, "*.py")) + glob.glob(os.path.join(root, "tools/*.py")):
        if not f.endswith("reference_flags_table.py"):
            text = open(f).read()
            if f.endswith("reference_flags.py"):
                text = text[text.index("def apply_reference_compat"):]          # the dictionaries themselves do not count as a use
            src += text
    read = set(re.findall(r"args\.([a-z_0-9]+)", src)) | set(re.findall(r"""["']([a-z_0-9]+)["']""", src))      # attribute reads and names passed to getattr / loops
    missing = sorted(d for d in rf.WIRED if d not in read)
    assert not missing, f"listed as wired but never read: {missing}"
    base = ["--num-layers", "2", "--hidden-size", "64", "--num-attention-heads", "4", "--micro-batch-size", "1", "--seq-length", "32", "--vocab-size", "128"]
    args = parse_args(base + ["--tp-size", "2", "--no-rope-fusion", "--multi-latent-attention", "--q-lora-rank", "32", "--kv-lora-rank", "16", "--qk-head-dim", "16",
                              "--qk-pos-emb-head-dim", "8", "--v-head-dim", "16", "--yarn-beta-fast", "16", "--ddp-average-in-collective", "--ddp-pad-buckets-for-high-nccl-busbw",
                              "--checkpoint-activations", "--grad-reduce-in-bf16", "--openai-gelu", "--bf16"])
    assert args.tensor_model_parallel_size == 2 and args.recompute_granularity == "full" and args.accumulate_allreduce_grads_in_fp32 is False
    validate_args(args, world_size=2)
    cfg = core_transformer_config_from_args(args)
    assert type(cfg).__name__ == "MLATransformerConfig" and (cfg.q_lora_rank, cfg.kv_lora_rank, cfg.qk_head_dim, cfg.qk_pos_emb_head_dim, cfg.v_head_dim, cfg.beta_fast) == (32, 16, 16, 8, 16, 16)
    assert cfg.apply_rope_fusion is False and abs(float(cfg.activation_func(torch.tensor(1.0))) - float(torch.nn.functional.gelu(torch.tensor(1.0), approximate="tanh"))) < 1e-7
    ddp = ddp_config_from_args(args)
    assert ddp.average_in_collective and ddp.pad_buckets_for_high_nccl_busbw and ddp.grad_reduce_in_fp32 is False
    assert parse_args(base).apply_rope_fusion is True                                              # the reference's command-line default
    # inert flags: reported, fatal when strict
    args = parse_args(base + ["--dino-head-hidden-size", "99"])
    assert rf.inert_flags_in_use(args, build_full_parser()) == ["--dino-head-hidden-size"]
    with pytest.raises(SystemExit):
        parse_args(base + ["--dino-head-hidden-size", "99", "--strict-reference-flags"])
    kw = rf.engine_kwargs_from_args(parse_args(base + ["--inference-dynamic-batching-block-size", "32", "--inference-max-requests", "8", "--enable-chunked-prefill",
                                                       "--inference-dynamic-batching-num-cuda-graphs", "4", "--inference-dynamic-batching-prefix-caching"]))
    assert kw == {"block_size": 32, "max_running": 8, "max_prefill_tokens_per_step": 2048, "enable_prefix_caching": True, "enable_cuda_graphs": True, "decode_batch_buckets": [2, 4, 6, 8]}


def test_step_batch_size_schedule_and_skipped_iterations_through_pretrain(tmp_path):
    """``--step-batch-size-schedule`` (token thresholds) drives the global batch size, ``--train-samples`` is converted to iterations against it and
    ``--iterations-to-skip`` consumes the data of an iteration without training on it (reference ``training.py:2155`` / ``:4648``)."""
    import re
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, os.path.join(root, "pretrain_gpt.py"), "--num-layers", "1", "--hidden-size", "32", "--num-attention-heads", "2", "--ffn-hidden-size", "64", "--seq-length", "32",
           "--max-position-embeddings", "32", "--micro-batch-size", "2", "--lr", "1e-3", "--lr-decay-samples", "100", "--lr-warmup-samples", "4", "--mock-data", "--tokenizer-type",
           "NullTokenizer", "--vocab-size", "127", "--log-interval", "1", "--distributed-backend", "gloo", "--eval-iters", "0", "--seed", "1234", "--step-batch-size-schedule", "0:2 256:4",
           "--train-samples", "24", "--iterations-to-skip", "3", "--train-sync-interval", "2", "--empty-unused-memory-level", "2", "--strict-reference-flags"]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env={**os.environ, "CUDA_VISIBLE_DEVICES": "", "MASTER_ADDR": "127.0.0.1", "MASTER_PORT": "29741"}, cwd=str(tmp_path))
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    rows = re.findall(r"iteration\s+(\d+)/\s+(\d+) \| consumed samples:\s+(\d+).*?global batch size:\s+(\d+)", r.stdout)
    assert [(int(i), int(c), int(b)) for i, _, c, b in rows] == [(1, 2, 2), (2, 4, 2), (4, 8, 2), (5, 12, 4), (6, 16, 4), (7, 20, 4), (8, 24, 4)]
    assert all(int(n) == 8 for _, n, _, _ in rows)


def test_fault_injector_from_reference_flags():
    import argparse

    from megatron_b200.core.fault_injector import Fault, FaultInjector, FaultInjectorConfig, InjectedFaultError

    assert FaultInjectorConfig.from_args(argparse.Namespace(), 4) is None
    ns = argparse.Namespace(fault_injector_fault_types="workload_exc,sigterm", fault_injector_fault_probabilities="1.0,0.0", fault_injector_ranks="0,2", fault_injector_fault_delay=0.05,
                            fault_injector_delay_start_iteration=3, fault_injector_seed=7)
    cfg = FaultInjectorConfig.from_args(ns, 4)
    assert cfg.fault_type == Fault.WORKLOAD_EXC and list(cfg.ranks) == [0, 2] and cfg.start_iteration == 3 and cfg.delay_s == pytest.approx(0.05)
    inj = FaultInjector(cfg, rank=2, world_size=4)
    inj.on_iteration(1)
    time.sleep(0.15)
    inj.on_iteration(2)                                   # the countdown has not started yet
    inj.on_iteration(3)
    time.sleep(0.3)
    with pytest.raises(InjectedFaultError):
        inj.on_iteration(4)
    assert not FaultInjector(cfg, rank=1, world_size=4).armed
    picks = FaultInjectorConfig.from_args(argparse.Namespace(fault_injector_fault_types="gpu_sleep", fault_injector_num_ranks=2, fault_injector_mtti_seconds=100.0, fault_injector_offset_seconds=5.0), 8)
    assert len(picks.ranks) == 2 and picks.delay_s > 5.0 and picks == FaultInjectorConfig.from_args(
        argparse.Namespace(fault_injector_fault_types="gpu_sleep", fault_injector_num_ranks=2, fault_injector_mtti_seconds=100.0, fault_injector_offset_seconds=5.0), 8)


def test_tokenizer_flags_and_vocab_padding():
    import argparse

    from megatron_b200.core.tokenizers import build_tokenizer_from_args
    from megatron_b200.core.tokenizers.text.tiktoken_tokenizer import compile_pattern
    from megatron_b200.training.arguments import parse_args, validate_args

    tok = build_tokenizer_from_args(argparse.Namespace(tokenizer_type="NullTokenizer", vocab_size=100, null_tokenizer_eod_id=7, null_tokenizer_pad_id=3))
    assert tok.eod == 7 and tok.pad == 3 and tok.vocab_size == 101
    assert build_tokenizer_from_args(argparse.Namespace(tokenizer_type="NullTokenizer", vocab_size=100)).eod == 100
    # the named splitters keep case runs / digits apart the way the reference patterns do
    assert compile_pattern("v1").findall("Hello world's 123") == ["Hello", " world", "'s", " ", "1", "2", "3"]
    assert compile_pattern("v2").findall("helloWorld HTTPServer") == ["hello", "World", " HTTPServer"]
    base = ["--num-layers", "1", "--hidden-size", "32", "--num-attention-heads", "2", "--seq-length", "16", "--max-position-embeddings", "16", "--micro-batch-size", "1", "--vocab-size", "1000"]
    a = validate_args(parse_args(base + ["--vocab-extra-ids", "5", "--make-vocab-size-divisible-by", "128"]), world_size=1)
    assert a.padded_vocab_size == 1024
    assert validate_args(parse_args(base + ["--no-pad-vocab-size"]), world_size=1).padded_vocab_size == 1000
    assert validate_args(parse_args(base + ["--padded-vocab-size", "2048"]), world_size=1).padded_vocab_size == 2048
    with pytest.raises(ValueError):
        validate_args(parse_args(base + ["--step-batch-size-schedule", "0:8", "--global-batch-size", "8"]), world_size=1)
    assert validate_args(parse_args(base + ["--step-batch-size-schedule", "0:8 1K:16"]), world_size=1).global_batch_size == 16


def test_every_flag_of_the_reference_runtime_parser_is_accepted():
    """Each option string of the reference's REAL parser (dataclass-generated groups included; stored in ``tests/golden/reference/training.json``) parses here
    with the same arity."""
    ref = [{"flags": flags, "nargs": nargs} for flags, nargs in _reference_golden("training.json")["parser_flags"]]
    assert len(ref) > 700
    from megatron_b200.training.arguments import build_full_parser

    ours = {f: a for a in build_full_parser()._actions for f in a.option_strings}
    missing = [f for r in ref for f in r["flags"] if f not in ours]
    assert not missing, missing
    arity = [(r["flags"][0], r["nargs"], ours[r["flags"][0]].nargs) for r in ref if (r["nargs"] == 0) != (ours[r["flags"][0]].nargs == 0)]
    assert not arity, arity
