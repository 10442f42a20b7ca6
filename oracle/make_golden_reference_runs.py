"""TEST INFRASTRUCTURE — golden data from runs of the UNMODIFIED reference, so that the tests compare against it without the
reference tree:
  * tests/golden/index_builders_random.json — digests of what its C++ index builders (oracle/_ref/, oracle/build_ref.sh) return
    on the randomised inputs of index_builder_cases.random_cases, and the schedule its BlendableDataset class (on those builders)
    gives the three-way blend of tests/test_index_builders_cpu.py;
  * tests/golden/erlangshen_script_batch.npz — the batch the ErLangShenCollator of
    fengshen/examples/pretrain_erlangshen_bert/pretrain_erlangshen.py, imported under fsb200.launch, builds from the first four
    rows of the tests' corpus fixture (tests/hf_fixtures.py) with np.random.RandomState(5) and a sorted vocabulary list.
Run:  FSB_REFERENCE_ROOT=<reference checkout> sh oracle/build_ref.sh && python oracle/make_golden_reference_runs.py <reference checkout>"""
import importlib.util
import json
import os
import runpy
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
GOLDEN = os.path.join(ROOT, "tests", "golden")


def erlangshen_batch(ref_root):
    sys.path[:0] = [os.path.join(ROOT, "tests"), os.path.join(ROOT, "fengshen-lm_b200")]
    import hf_fixtures as F
    from fsb200 import launch
    script = os.path.join(ref_root, "fengshen", "examples", "pretrain_erlangshen_bert", "pretrain_erlangshen.py")
    launch.prepare(script)
    ns = runpy.run_path(script, run_name="reference_not_main")
    with tempfile.TemporaryDirectory() as tmp:
        F.bert_dir(os.path.join(tmp, "m"))
        rows = [json.loads(line) for line in open(F.bert_corpus(os.path.join(tmp, "train.json")), encoding="utf8")][:4]
        tok = ns["AutoTokenizer"].from_pretrained(os.path.join(tmp, "m"))
        coll = ns["ErLangShenCollator"](tokenizer=tok, max_seq_length=64, masked_lm_prob=0.15)
        coll.setup()
        coll.np_rng = np.random.RandomState(5)
        coll.vocab_id_list = sorted(coll.vocab_id_list)
        return {k: v.numpy() for k, v in coll(rows).items()}


def index_builders(ref_root):
    sys.path.insert(0, HERE)
    import index_builder_cases as C
    from make_golden_index_builders import load_reference_helpers, quiet_stdout
    import torch.distributed as dist
    ref = load_reference_helpers()
    if ref is None:
        raise SystemExit("oracle/_ref/helpers*.so missing: run `sh oracle/build_ref.sh` first")
    with quiet_stdout():
        out = {k: C.digest(v) for k, v in C.random_cases(ref).items()}
    # the reference class imports `helpers` from its package at call time: point that name at the reference's own build
    import fengshen.data.megatron_dataloader as pkg
    sys.modules["fengshen.data.megatron_dataloader.helpers"] = pkg.helpers = ref
    spec = importlib.util.spec_from_file_location(
        "ref_blendable_dataset", os.path.join(ref_root, "fengshen", "data", "megatron_dataloader", "blendable_dataset.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    dist.init_process_group("gloo", init_method="tcp://127.0.0.1:29632", rank=0, world_size=1)   # it calls get_rank()
    with quiet_stdout():
        bd = mod.BlendableDataset([list(range(70)), list(range(20)), list(range(10))], [7, 2, 1])
    dist.destroy_process_group()
    out["blendable_dataset_index"] = bd.dataset_index.tolist()
    out["blendable_dataset_sample_index"] = bd.dataset_sample_index.tolist()
    return out


def main():
    if len(sys.argv) != 2 or not os.path.isdir(os.path.join(sys.argv[1], "fengshen")):
        raise SystemExit("usage: python oracle/make_golden_reference_runs.py <reference checkout>")
    ref_root = sys.argv[1]
    path = os.path.join(GOLDEN, "erlangshen_script_batch.npz")
    np.savez_compressed(path, **erlangshen_batch(ref_root))
    print(path, os.path.getsize(path), "bytes")
    path = os.path.join(GOLDEN, "index_builders_random.json")
    with open(path, "w") as f:
        json.dump(index_builders(ref_root), f, indent=0, sort_keys=True)
    print(path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
