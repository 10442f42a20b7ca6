"""CPU: the host side of the HF-backed recipes end to end — fsb200.launch, transformers rebinding, example script, compat
Trainer, ZeroEngine (ZeRO-1 + clipping / default strategy), DeepSpeed-layout checkpoints, resume (step / sample / LR-schedule
position), metric-formatted checkpoint names, HF-style export — with the model classes replaced by tests/toy_models.py and the
engine kernels by tests/cpu_kernels.py. The bodies are the ones tests/test_hf_scripts_gpu.py runs on the real models."""
import os
import sys

import pytest

import hf_fixtures as F
import hf_recipes as R

for p in ("fengshen-lm_b200",):
    if os.path.join(F.ROOT, p) not in sys.path:
        sys.path.insert(0, os.path.join(F.ROOT, p))


@pytest.fixture
def launched_with_doubles(monkeypatch):
    saved_path = list(sys.path)
    for k in [k for k in sys.modules if k.split(".")[0] in ("fengshen", "pytorch_lightning", "deepspeed")]:
        monkeypatch.delitem(sys.modules, k)
    import cpu_kernels
    import fsb200.engine as engine
    import fsb200.hf as hf
    import fsb200.launch as launch
    import toy_models as T

    class CpuEngine(engine.ZeroEngine):
        def __init__(self, model, **kw):
            kw.setdefault("kernels", cpu_kernels)
            super().__init__(model, **kw)

    monkeypatch.setattr(engine, "ZeroEngine", CpuEngine)
    monkeypatch.setattr(hf, "MegatronBertForPreTraining",
                        type("MegatronBertForPreTraining", (hf._HFSurface, T.ToyMegatronBert), {"config_name": "MegatronBertConfig"}))
    monkeypatch.setattr(hf, "GPT2LMHeadModel",
                        type("GPT2LMHeadModel", (hf._HFSurface, T.ToyGPT2), {"config_name": "GPT2Config"}))
    launch.prepare(R.EXAMPLE)
    yield hf
    hf.uninstall()
    sys.path[:] = saved_path


def test_erlangshen_recipe_host_flow(launched_with_doubles, tmp_path, monkeypatch):
    trainer, module = R.erlangshen_recipe(tmp_path, monkeypatch, min_drop=0.05, lr="2e-2")
    assert not module.model.flat.params.is_cuda


def test_wenzhong_recipe_host_flow(launched_with_doubles, tmp_path):
    R.wenzhong_recipe(tmp_path, min_drop=0.02, device="cpu")


# ---- two data-parallel ranks over gloo: sharded optimizer state, per-rank sample streams, two optimizer-shard files, resume ----
def _rank_main(rank, world, port, workdir, q):
    import json
    import runpy
    os.environ.update(RANK=str(rank), LOCAL_RANK=str(rank), WORLD_SIZE=str(world), MASTER_ADDR="127.0.0.1",
                      MASTER_PORT=str(port), PL_DEEPSPEED_CONFIG_PATH=os.path.join(workdir, "ds_config.json"))
    sys.path.insert(0, os.path.join(F.ROOT, "tests"))
    sys.path.insert(0, os.path.join(F.ROOT, "fengshen-lm_b200"))
    import torch
    import cpu_kernels
    import fsb200.engine as engine
    import fsb200.hf as hf
    import fsb200.launch as launch
    import toy_models as T

    class CpuEngine(engine.ZeroEngine):
        def __init__(self, model, **kw):
            kw.setdefault("kernels", cpu_kernels)
            super().__init__(model, **kw)

    engine.ZeroEngine = CpuEngine
    hf.MegatronBertForPreTraining = type("MegatronBertForPreTraining", (hf._HFSurface, T.ToyMegatronBert),
                                         {"config_name": "MegatronBertConfig"})
    launch.prepare(R.EXAMPLE)
    ns = runpy.run_path(R.EXAMPLE, run_name="example_not_main")

    def argv(epochs):
        return ["--model_path", os.path.join(workdir, "m"), "--train_file", os.path.join(workdir, "train.json"),
                "--train_batchsize", "4", "--max_seq_length", "64", "--max_epoch", str(epochs), "--learning_rate", "2e-2",
                "--strategy", "deepspeed_stage_1", "--replace_sampler_ddp", "False", "--dataloader_workers", "0",
                "--log_every_n_steps", "1", "--default_root_dir", workdir, "--save_ckpt_path", os.path.join(workdir, "ckpt"),
                "--load_ckpt_path", os.path.join(workdir, "ckpt", "last.ckpt"), "--save_last", "--precision", "bf16",
                "--native_collator"]              # sample assembly through fsb_bert_collate in this (two-rank) variant

    trainer, module = ns["main"](argv(1))
    first = (trainer.global_step, trainer.engine.world, module.model.flat.world_size, module.model.flat.params.float().numpy().copy())
    trainer2, module2 = ns["main"](argv(2))
    q.put((rank, first, (trainer2.global_step, getattr(module2, "consumed_samples", None),
                         module2.model.flat.params.float().numpy().copy())))
    torch.distributed.barrier()
    torch.distributed.destroy_process_group()


def test_erlangshen_recipe_two_ranks_over_gloo(tmp_path, monkeypatch):
    import json
    import numpy as np
    import torch
    import torch.multiprocessing as mp
    # the ranks inherit this: they take the host path (gloo, CPU kernels) on machines with a GPU too, where the compat Trainer
    # would otherwise bind rank r to cuda:r over NCCL
    monkeypatch.setenv("CUDA_VISIBLE_DEVICES", "")
    F.bert_dir(tmp_path / "m")
    F.bert_corpus(tmp_path / "train.json", n=64)
    (tmp_path / "ds_config.json").write_text(json.dumps({"zero_optimization": {"stage": 1}, "bf16": {"enabled": True},
                                                         "gradient_clipping": 2, "train_micro_batch_size_per_gpu": 4}))
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_rank_main, args=(r, 2, 29655, str(tmp_path), q)) for r in range(2)]
    for p in procs:
        p.start()
    try:
        got = {}
        for _ in range(2):
            rank, first, second = q.get(timeout=240)
            got[rank] = (first, second)
    finally:
        for p in procs:
            p.join(timeout=60)
            if p.is_alive():
                p.terminate()
    assert all(p.exitcode == 0 for p in procs)
    for rank in (0, 1):
        (steps, eng_world, flat_world, _), (steps2, consumed, _) = got[rank]
        assert (steps, eng_world, flat_world) == (8, 2, 2)            # 64 documents / (4 per rank x 2 ranks)
        assert steps2 == 16 and consumed == 64                        # resumed: 8 + 8 steps, sample counter from the checkpoint
    assert np.array_equal(got[0][0][3], got[1][0][3]) and np.array_equal(got[0][1][2], got[1][1][2])   # ranks agree after all-gather
    assert not np.array_equal(got[0][0][3], got[0][1][2])
    ck = tmp_path / "ckpt" / "last.ckpt" / "checkpoint"
    assert sorted(os.listdir(ck)) == ["mp_rank_00_model_states.pt", "zero_pp_rank_0_mp_rank_00_optim_states.pt",
                                      "zero_pp_rank_1_mp_rank_00_optim_states.pt"]
    state = torch.load(ck / "mp_rank_00_model_states.pt", map_location="cpu", weights_only=False)
    assert state["global_step"] == 16 and state["global_samples"] == 128
    shard = torch.load(ck / "zero_pp_rank_1_mp_rank_00_optim_states.pt", map_location="cpu", weights_only=False)
    assert shard["format"] == "fsb200-zero-shard-v1"


def test_t5_recipe_host_flow(launched_with_doubles, tmp_path, monkeypatch):
    import fsb200.hf as hf
    import toy_models as T
    import transformers
    toy = type("MT5ForConditionalGeneration", (hf._HFSurface, T.ToyMT5), {"config_name": "MT5Config"})
    monkeypatch.setattr(hf, "MT5ForConditionalGeneration", toy)
    hf.install()
    assert transformers.MT5Tokenizer is transformers.T5Tokenizer                # the alias transformers 4.x shipped
    R.t5_recipe(tmp_path, min_drop=None, lr="2e-2")


def test_gradient_accumulation_through_the_trainer(launched_with_doubles, tmp_path, monkeypatch):
    """--accumulate_grad_batches 2 with ZeRO-2 (fp32 shard accumulation in the engine): optimizer steps = micro-batches / 2, the
    step arithmetic of get_total_steps and the checkpoint's sample counter follow (model_utils.py:194-209, SURVEY §3.4)."""
    import json
    import runpy
    import torch
    F.bert_dir(tmp_path / "m")
    corpus = F.bert_corpus(tmp_path / "train.json", n=64)
    monkeypatch.delenv("PL_DEEPSPEED_CONFIG_PATH", raising=False)
    ns = runpy.run_path(R.EXAMPLE, run_name="example_not_main")
    trainer, module = ns["main"](["--model_path", str(tmp_path / "m"), "--train_file", str(corpus), "--train_batchsize", "4",
                                  "--max_seq_length", "64", "--max_epochs", "1", "--accumulate_grad_batches", "2",
                                  "--learning_rate", "2e-2", "--strategy", "deepspeed_stage_2", "--gradient_clip_val", "1.0",
                                  "--replace_sampler_ddp", "False", "--dataloader_workers", "0", "--log_every_n_steps", "1",
                                  "--default_root_dir", str(tmp_path), "--save_ckpt_path", str(tmp_path / "ckpt"),
                                  "--load_ckpt_path", str(tmp_path / "ckpt" / "last.ckpt"), "--save_last", "--native_collator"])
    assert module.total_steps == 8 and trainer.global_step == 8               # 64 documents / 4 per micro-batch / 2
    eng = trainer.engine
    assert eng.ga_steps == 2 and eng.stage == 2 and eng.acc32 is not None and eng.grad_clip == 1.0
    assert module.model.loss_scale == 0.5                                       # 1 / (world x GA): the mean over micro-batches
    state = torch.load(tmp_path / "ckpt" / "last.ckpt" / "checkpoint" / "mp_rank_00_model_states.pt", map_location="cpu",
                       weights_only=False)
    assert state["global_step"] == 8 and state["global_samples"] == 64
    losses = R.losses_of(trainer)
    assert len(losses) == 8 and losses[-1] < losses[0]
