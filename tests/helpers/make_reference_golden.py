"""Regenerate ``tests/golden/reference/``: what the UNMODIFIED reference computes for the inputs of the reference-parity tests (run as a script).

Needs the reference installed under ``baseline/_ref`` (``pip install --no-deps --no-build-isolation --target baseline/_ref <reference checkout>``); the
tests themselves only read the stored files.

    python tests/helpers/make_reference_golden.py

Model runs (loss and gradients of tiny models, three optimizer steps) keep, per tensor, its shape, max |x|, sum, L2 norm and the values at a fixed
sample of flat indices, so that every file stays small; the parity tests check each of those against this framework's full tensors.
"""
import json
import os
import shutil
import socket
import subprocess
import sys
import tempfile
import zlib

import numpy as np
import torch

REPO = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
TESTS = os.path.join(REPO, "tests")
REF = os.path.join(REPO, "baseline", "_ref")
OUT = os.path.join(TESTS, "golden", "reference")
SAMPLES = 8

sys.path.insert(0, TESTS)
sys.path.insert(0, REPO)


def _f32(x):
    """Shortest decimal that reads back as the same float32."""
    return float(str(np.float32(x)))


def compact_tensor(name, t):
    t = t.detach().float().cpu()
    flat = t.flatten()
    n = flat.numel()
    idx = sorted(np.random.default_rng(zlib.crc32(name.encode())).choice(n, size=min(n, SAMPLES), replace=False).tolist())
    d = flat.double()
    return {"shape": list(t.shape), "absmax": float(d.abs().max()), "sum": float(d.sum()), "norm": float(d.norm()), "idx": idx, "val": [_f32(flat[i]) for i in idx]}


def compact(result):
    out = {}
    for k, v in result.items():
        if isinstance(v, dict):
            out[k] = {n: compact_tensor(n, t) for n, t in v.items()}
        elif isinstance(v, tuple):
            out[k] = list(v)
        else:
            out[k] = v
    return out


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def run_reference_model(tmp, tp, variant="", world=None, extra=(), env_extra=None):
    """Spawn ``ref_cpu_model.py`` on ``world`` gloo ranks; returns the per-rank results it saved."""
    world = world or tp
    port = _free_port()
    prefix = os.path.join(tmp, f"ref_{variant or 'gpt'}_{'_'.join(extra[:1])}_tp{tp}")
    procs = []
    for r in range(world):
        env = dict(os.environ, RANK=str(r), WORLD_SIZE=str(world), MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), OMP_NUM_THREADS="1", REF_VARIANT=variant,
                   **(env_extra or {}))
        procs.append(subprocess.Popen([sys.executable, os.path.join(TESTS, "helpers", "ref_cpu_model.py"), prefix, str(tp), *extra], env=env,
                                      stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True))
    for p in procs:
        out, _ = p.communicate(timeout=600)
        assert p.returncode == 0, out[-3000:]
    if extra and extra[0] == "save":
        return None
    return [torch.load(f"{prefix}.rank{r}.pt") for r in range(world)]


def write_json(name, obj):
    with open(os.path.join(OUT, name), "w") as f:
        json.dump(obj, f, separators=(",", ":"))
        f.write("\n")


# name: (tp, REF_VARIANT, world size, extra environment)
MODEL_RUNS = {
    "gpt_tp1": (1, "", 1, {}),
    "gpt_tp2": (2, "", 2, {}),
    "moe": (1, "moe", 1, {}),
    "moe_dsv3": (1, "moe_dsv3", 1, {}),
    "moe_drop": (1, "moe_drop", 1, {}),
    "moe_ep2": (1, "moe_ep2", 2, {}),
    "mup": (1, "", 1, {"REF_CFG_OVERRIDE": '{"use_mup": true, "mup_base_hidden_size": 32, "mup_embedding_mult": 2.0}'}),
    "bert": (1, "bert", 1, {}),
    "t5": (1, "t5", 1, {}),
    "vit": (1, "vit", 1, {}),
    "optim": (1, "optim", 1, {}),
    "distopt": (1, "distopt", 2, {}),
    "pp2": (1, "pp2", 2, {}),
}


def models(tmp):
    for name, (tp, variant, world, env) in MODEL_RUNS.items():
        ranks = run_reference_model(tmp, tp, variant, world, env_extra=env)
        write_json(f"model_{name}.json", [compact(r) for r in ranks])
        print("model", name)


def checkpoints(tmp):
    """The reference's own torch_dist checkpoints of the (smaller) interop model, written at TP 1 and TP 2, as reproducible tarballs."""
    import gzip
    import tarfile

    from test_reference_parity_cpu import CKPT_MODEL

    for tp in (1, 2):
        src = os.path.join(tmp, f"ckpt_tp{tp}")
        os.makedirs(src)
        run_reference_model(tmp, tp, extra=("save", src), env_extra={"REF_MODEL_SIZE": json.dumps(CKPT_MODEL)})
        with gzip.GzipFile(os.path.join(OUT, f"ckpt_tp{tp}.tar.gz"), "wb", compresslevel=9, mtime=0) as gz, tarfile.open(fileobj=gz, mode="w") as tar:
            for name in sorted(os.listdir(src)):
                info = tar.gettarinfo(os.path.join(src, name), arcname=name)
                info.mtime, info.uid, info.gid, info.uname, info.gname = 0, 0, 0, "", ""
                with open(os.path.join(src, name), "rb") as f:
                    tar.addfile(info, f)
        print("checkpoint tp", tp, sorted(os.listdir(src)))


def datasets(tmp):
    from test_reference_parity_cpu import DATA_COUNTS, DATA_SEED, DATA_SEQ, DATA_SPLIT, data_blend_args, write_corpora

    for blend in (False, True):
        d = os.path.join(tmp, f"data_{blend}")
        os.makedirs(d)
        write_corpora(d)
        out = os.path.join(d, "ref.pt")
        r = subprocess.run([sys.executable, os.path.join(TESTS, "helpers", "ref_data.py"), out, os.path.join(d, "ref_cache"), str(DATA_SEQ), str(DATA_SEED), DATA_SPLIT,
                            *map(str, DATA_COUNTS), *data_blend_args(d, blend)], env=dict(os.environ, OMP_NUM_THREADS="1"), capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-3000:]
        ref = torch.load(out)
        dump = {}
        for split, v in ref.items():
            dump[split] = None if v is None else {"len": v["len"], "samples": {str(i): {k: [str(t.dtype).replace("torch.", ""), t.tolist()] for k, t in s.items()}
                                                                               for i, s in v["samples"].items()}}
        write_json(f"gpt_dataset_{'blend' if blend else 'single'}.json", dump)
        print("dataset blend", blend)


def pure():
    r = subprocess.run([sys.executable, os.path.join(TESTS, "helpers", "ref_pure.py")], cwd=tempfile.gettempdir(), capture_output=True, text=True, timeout=600)
    line = [ln for ln in r.stdout.splitlines() if ln.startswith("JSON:")]
    assert line, r.stdout[-2000:] + r.stderr[-2000:]
    write_json("schedules_and_ranks.json", json.loads(line[0][5:]))
    print("pure")


def _with_reference(fn):
    sys.path.insert(0, REF)
    saved = {k: v for k, v in sys.modules.items() if k == "megatron" or k.startswith("megatron.")}
    try:
        return fn()
    finally:
        sys.path.remove(REF)
        for k in [k for k in sys.modules if k == "megatron" or k.startswith("megatron.")]:
            del sys.modules[k]
        sys.modules.update(saved)


def value_parity():
    import test_reference_value_parity_cpu as T

    def run():
        from megatron.core.models.hybrid import hybrid_layer_allocation
        from megatron.core.transformer.experimental_attention_variant import dsa_indexer_loss, dsa_masking
        from megatron.core.transformer.moe import moe_utils

        return {"dsa_indexer_loss": T._indexer_loss_outputs(dsa_indexer_loss), "dsa_masking": T._masking_outputs(dsa_masking, torch.device("cpu")),
                "moe_routing_scores": T._routing_scores_outputs(moe_utils), "hybrid_layer_allocation": T._hybrid_outputs(hybrid_layer_allocation)}

    torch.save(_with_reference(run), os.path.join(OUT, "value_parity.pt"))
    print("value parity")


def _flops_args(**k):
    import argparse

    d = dict(seq_length=8192, hidden_size=4096, num_layers=32, ffn_hidden_size=14336, num_attention_heads=32, group_query_attention=True, num_query_groups=8, kv_channels=128,
             padded_vocab_size=128256, swiglu=True, num_experts=None, moe_layer_freq=1, moe_router_topk=1, moe_ffn_hidden_size=None, moe_latent_size=None,
             moe_shared_expert_intermediate_size=None, mtp_num_layers=None, multi_latent_attention=False, experimental_attention_variant=None, attention_output_gate=False,
             hybrid_layer_pattern=None)
    d.update(k)
    return argparse.Namespace(**d)


def _reference_flops_fn():
    """The reference's analytic model, extracted from its training loop's source (pure python)."""
    import ast

    src = open(os.path.join(REF, "megatron", "training", "training.py")).read()
    fn = [n for n in ast.parse(src).body if isinstance(n, ast.FunctionDef) and n.name == "num_floating_point_operations"][0]
    ns = {}
    exec("def is_linear_attention_variant(v): return v in ('gdn', 'gdn2', 'gated_delta_net')\n"
         "def is_gated_delta_net_variant(v): return v in ('gdn', 'gdn2', 'gated_delta_net')\n"
         "def is_hybrid_model(args): return False\n" + ast.get_source_segment(src, fn), ns)
    return ns["num_floating_point_operations"]


def training():
    from test_training_utils_cpu import FLOPS_CASES

    sys.path.insert(0, os.path.join(REPO, "tools"))
    from gen_reference_flag_table import _introspect

    ref = _reference_flops_fn()
    flops = {name: ref(_flops_args(**ref_kw), batch, **call_kw) for name, (_, ref_kw, batch, call_kw) in FLOPS_CASES.items()}
    flags = [[r["flags"], r["nargs"]] for r in _introspect(REF)]
    assert len(flags) > 700
    write_json("training.json", {"flops": flops, "parser_flags": flags})
    print("training")


def integrity(tmp):
    from test_utils_additions_cpu import INTEGRITY_FILES

    d = os.path.join(tmp, "integrity")
    os.makedirs(d)
    for name, data in INTEGRITY_FILES.items():
        with open(os.path.join(d, name), "wb") as f:
            f.write(data)

    def run():
        from megatron.core.dist_checkpointing.validation import save_integrity_manifest

        save_integrity_manifest(d)

    _with_reference(run)
    shutil.copyfile(os.path.join(d, "integrity.json"), os.path.join(OUT, "integrity.json"))
    print("integrity")


def main():
    assert os.path.isdir(os.path.join(REF, "megatron", "core")), f"the reference is not installed under {REF}"
    os.makedirs(OUT, exist_ok=True)
    with tempfile.TemporaryDirectory() as tmp:
        value_parity()
        integrity(tmp)
        training()
        pure()
        datasets(tmp)
        checkpoints(tmp)
        models(tmp)


if __name__ == "__main__":
    main()
