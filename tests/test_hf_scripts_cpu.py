"""CPU half of the HF-backed recipes (C2 / C3; SURVEY §8a row A16, §8f rank 3): everything the scripts do before the model
touches CUDA — the launcher's sys.path / transformers rebinding, argument parsers, tokenizer, collator, data modules, batches —
for fsb200's own example script, checked against the batch the UNMODIFIED reference script
(examples/pretrain_erlangshen_bert/pretrain_erlangshen.py) builds, recorded as golden data. Building a model without a GPU must
fail loudly (no CPU fallback on the product path)."""
import argparse
import os
import runpy
import sys

import numpy as np
import pytest
import torch

import hf_fixtures as F

ROOT = F.ROOT
EXAMPLE = os.path.join(ROOT, "examples", "pretrain_erlangshen_bert.py")


@pytest.fixture
def launcher(monkeypatch):
    """fsb200.launch.prepare(script) with everything it touches restored afterwards."""
    monkeypatch.syspath_prepend(os.path.join(ROOT, "fengshen-lm_b200"))
    saved_path = list(sys.path)
    for k in [k for k in sys.modules if k.split(".")[0] in ("fengshen", "pytorch_lightning", "deepspeed")]:
        monkeypatch.delitem(sys.modules, k)
    import fsb200.hf as hf
    import fsb200.launch as launch

    def prepare(script):
        launch.prepare(script)
        return hf
    yield prepare
    hf.uninstall()
    sys.path[:] = saved_path


def test_install_rebinds_transformers_names_and_uninstall_restores(launcher):
    hf = launcher(EXAMPLE)
    from transformers import BertForMaskedLM, GPT2LMHeadModel, MegatronBertForPreTraining, MT5ForConditionalGeneration
    for c in (BertForMaskedLM, GPT2LMHeadModel, MegatronBertForPreTraining, MT5ForConditionalGeneration):
        assert c.__module__ == "fsb200.hf", c
    import fengshen
    assert os.path.join("fengshen-lm_b200", "compat") in fengshen.__file__
    hf.uninstall()
    from transformers import GPT2LMHeadModel as G2
    assert G2.__module__.startswith("transformers.")


def test_hf_named_classes_fail_loudly(launcher, tmp_path):
    hf = launcher(EXAMPLE)
    with pytest.raises(FileNotFoundError, match="not a local directory"):
        hf.GPT2LMHeadModel.from_pretrained("IDEA-CCNL/Wenzhong-GPT2-110M")
    F.bert_dir(tmp_path / "m")
    with pytest.raises(FileNotFoundError, match="pytorch_model.bin"):
        hf.MegatronBertForPreTraining.from_pretrained(str(tmp_path / "m"))
    if not torch.cuda.is_available():
        from transformers import MegatronBertConfig
        with pytest.raises(RuntimeError, match="CUDA|NVIDIA"):
            hf.MegatronBertForPreTraining(MegatronBertConfig.from_pretrained(str(tmp_path / "m")))


def _erlangshen_args(ns, tmp, mdir, corpus, extra=()):
    p = argparse.ArgumentParser()
    p = ns["add_module_args"](p)
    p = ns["UniversalDataModule"].add_data_specific_args(p)
    p = ns["Trainer"].add_argparse_args(p)
    p = ns["ErLangShenBert"].add_module_specific_args(p)
    p = ns["UniversalCheckpoint"].add_argparse_args(p)
    return p.parse_args(["--model_path", str(mdir), "--train_file", str(corpus), "--val_file", str(corpus), "--test_file",
                         str(corpus), "--train_batchsize", "4", "--max_seq_length", "64", "--max_epoch", "1",
                         "--dataloader_workers", "0", "--default_root_dir", str(tmp), "--save_ckpt_path", str(tmp / "ckpt"),
                         "--load_ckpt_path", str(tmp / "ckpt" / "last.ckpt"), "--replace_sampler_ddp", "False", *extra])


def _check_mlm_batch(batch, B, L, tok):
    assert set(batch) == {"input_ids", "attention_mask", "token_type_ids", "labels", "next_sentence_label"}
    assert batch["input_ids"].shape == (B, L) and batch["labels"].shape == (B, L)
    assert batch["next_sentence_label"].shape == (B,) and batch["next_sentence_label"].dtype == torch.int64
    lab, ids, am = batch["labels"], batch["input_ids"], batch["attention_mask"]
    assert (ids[:, 0] == tok.cls_token_id).all()
    assert ((lab != -100) & (am == 0)).sum() == 0                 # never a target on padding
    n = (lab != -100).sum(1).numpy()
    assert (n >= 1).all() and (n <= np.ceil(0.15 * am.sum(1).numpy()) + 1).all()
    assert ((ids == tok.mask_token_id) & (lab != -100)).sum() > 0


def test_example_script_cpu_half(launcher, tmp_path):
    launcher(EXAMPLE)
    ns = runpy.run_path(EXAMPLE, run_name="example_not_main")
    assert ns["MegatronBertForPreTraining"].__module__ == "fsb200.hf"
    F.bert_dir(tmp_path / "m")
    corpus = F.bert_corpus(tmp_path / "train.json")
    args = _erlangshen_args(ns, tmp_path, tmp_path / "m", corpus)
    assert args.max_epochs == 1 and args.replace_sampler_ddp is False
    tok = ns["AutoTokenizer"].from_pretrained(args.model_path)
    coll = ns["ErLangShenCollator"](tokenizer=tok, max_seq_length=args.max_seq_length, masked_lm_prob=args.masked_lm_prob,
                                    content_key=args.sample_content_key)
    coll.setup()
    ds = ns["JsonLines"](args.train_file)
    dm = ns["UniversalDataModule"](tokenizer=tok, args=args, collate_fn=coll, datasets={"train": ds})
    _check_mlm_batch(coll([ds[i] for i in range(4)]), 4, 64, tok)
    # the Megatron sampler path (--replace_sampler_ddp False): a stub trainer is all get_custom_sampler needs
    from types import SimpleNamespace
    dm.trainer = SimpleNamespace(world_size=1, global_rank=0, global_step=0, accumulate_grad_batches=1, current_epoch=0,
                                 lightning_module=SimpleNamespace())
    batches = list(dm.train_dataloader())
    assert len(batches) == len(ds) // 4
    _check_mlm_batch(batches[0], 4, 64, tok)
    if not torch.cuda.is_available():
        with pytest.raises(RuntimeError, match="CUDA|NVIDIA"):
            ns["ErLangShenBert"](args, tokenizer=tok)


def test_unmodified_erlangshen_script_cpu_half(launcher, tmp_path, monkeypatch):
    """The MLM + SOP batch of the unmodified pretrain_erlangshen.py: its own ErLangShenCollator, run under fsb200.launch on the
    first four rows of this corpus (RandomState(5), sorted vocabulary), recorded in tests/golden/erlangshen_script_batch.npz by
    oracle/make_golden_reference_runs.py. The rows come through UniversalDataModule(--train_file ...) and `datasets`, as in the
    script; the library collator must reproduce the batch draw for draw."""
    import datasets
    monkeypatch.setattr(datasets.config, "HF_DATASETS_CACHE", str(tmp_path / "hf_datasets"))
    launcher(EXAMPLE)
    ns = runpy.run_path(EXAMPLE, run_name="example_not_main")
    assert os.path.join("fengshen-lm_b200", "compat") in sys.modules["fengshen.data.data_utils.mask_utils"].__file__
    F.bert_dir(tmp_path / "m")
    corpus = F.bert_corpus(tmp_path / "train.json")
    args = _erlangshen_args(ns, tmp_path, tmp_path / "m", corpus)
    tok = ns["AutoTokenizer"].from_pretrained(args.model_path)
    dm = ns["UniversalDataModule"](tokenizer=tok, args=args, collate_fn=None)        # --train_file through `datasets`
    ds = dm.datasets[args.train_datasets_field]
    rows = [ds[i] for i in range(4)]
    from fengshen.data.data_utils.collators import ErLangShenCollator as Lib
    lib = Lib(tokenizer=tok, max_seq_length=args.max_seq_length, masked_lm_prob=args.masked_lm_prob)
    lib.setup()
    lib.np_rng = np.random.RandomState(5)
    lib.vocab_id_list = sorted(lib.vocab_id_list)
    ours = lib(rows)
    _check_mlm_batch(ours, 4, 64, tok)
    theirs = np.load(os.path.join(ROOT, "tests", "golden", "erlangshen_script_batch.npz"))
    assert set(ours) == set(theirs.files)
    for k in theirs.files:
        assert ours[k].dtype == torch.from_numpy(theirs[k]).dtype and np.array_equal(ours[k].numpy(), theirs[k]), k


def _qa_args(parser_owner, tmp, mdir):
    p = argparse.ArgumentParser()
    p.add_argument('--do_eval_only', action='store_true', default=False)
    p.add_argument('--pretrained_model_path', default=str(mdir), type=str)
    p = parser_owner.add_data_specific_args(p)
    return p.parse_args(["--data_dir", str(tmp / "data"), "--train_batchsize", "4", "--valid_batchsize", "4",
                         "--max_seq_length", "64", "--num_workers", "0"])


def test_medical_qa_datamodule(launcher, tmp_path):
    launcher(EXAMPLE)
    from fengshen.data.task_dataloader.medicalQADataset import GPT2QADataModel
    F.gpt2_tokenizer_dir(tmp_path / "m")
    rows = F.qa_files(tmp_path / "data")
    dm = GPT2QADataModel(_qa_args(GPT2QADataModel, tmp_path, tmp_path / "m"))
    assert len(dm.train_data) == len(rows)
    b = next(iter(dm.val_dataloader()))
    assert b["input_ids"].shape == (4, 64) and b["question"][0] == rows[0]["Question"]
    pad = dm.train_data.tokenizer.pad_token_id
    assert ((b["labels"] == -100) == (b["input_ids"] == pad)).all()
    assert ((b["attention_mask"] == 0) <= (b["input_ids"] == pad)).all()
    n = int(b["attention_mask"][0].sum())
    text = rows[0]["Question"] + rows[0]["answer"]
    assert dm.train_data.tokenizer.decode(b["input_ids"][0, :n]) == text[:n]           # byte-level, ASCII: one token per char
