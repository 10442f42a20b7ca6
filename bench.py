#!/usr/bin/env python
"""bench.py — tokens/s of the data-parallel pretraining step (forward + backward + sharded AdamW) on synthetic tokens.

    python bench.py --gpus N --steps K --warmup W [--workload NAME] [--impl reference] [--dump-outputs DIR]

Workloads (BASELINE.json `configs`):
    gpt2-110m        C2  Wenzhong-GPT2-110M, seq 1024, 32 sequences per GPU, bf16            (default at any N; weak scaling)
    ziya-llama-13b   C4  Ziya-LLaMA-13B, seq 2048, 32 sequences per GPU, ZeRO-2, bf16        (needs >= 4 GPUs of HBM)
    ziya-llama-13b-L{n}  same width, n layers (NOT a BASELINE config; kernel bring-up / profiling only)
A "step" is one optimizer step over the per-GPU batch (micro-batches x gradient accumulation). `value` is whole-job
tokens/s with the token tensors already resident in HBM; `e2e` repeats the measurement through the public step API
(fsb200.trainer.PretrainStep.step) from pinned host memory, with the host->device copies and the loss read-back inside
the timed region. Timing: CUDA events, barrier + synchronize on both sides, max over ranks.
`--impl reference` times the reference's own CPU implementation of the same step on the host cores (see DESIGN.md).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "fengshen-lm_b200"))

import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

WORKLOADS = {
    # name: family, dims, seq, per-GPU sequences, micro-batch
    "gpt2-110m": dict(family="gpt2", vocab_size=50264, n_positions=1024, n_embd=768, n_layer=12, n_head=12, seq=1024,
                      per_gpu=32, micro=32, lr=1e-4, betas=(0.9, 0.999), wd=0.1, clip=0.0,
                      label="Wenzhong-GPT2-110M pretrain, seq 1024, batch 32/GPU (BASELINE configs[1])"),
    "bert-base": dict(family="bert", variant="bert", vocab_size=21128, hidden_size=768, num_hidden_layers=12,
                      num_attention_heads=12, intermediate_size=3072, hidden_act="gelu", seq=128, per_gpu=8, micro=8,
                      lr=1e-4, betas=(0.9, 0.999), wd=0.1, clip=0.0,
                      label="Erlangshen-BERT-base MLM, seq 128, batch 8 (BASELINE configs[0])"),
    "megatronbert-1.3b": dict(family="bert", variant="megatron", vocab_size=21128, hidden_size=2048,
                              num_hidden_layers=24, num_attention_heads=32, intermediate_size=8192, hidden_act="gelu",
                              seq=512, per_gpu=128, micro=32, lr=1e-4, betas=(0.9, 0.999), wd=0.1, clip=1.0, stage=1,
                              label="Erlangshen-MegatronBERT-1.3B MLM+SOP pretrain, seq 512, batch 128/GPU, ZeRO-1 "
                                    "(BASELINE configs[2])"),
    # Randeng-T5-784M = mT5-large shape (SURVEY.md §8 C5): d 1024, 24+24 layers, 16 heads x 64, gated-GeLU d_ff 2816; the
    # released vocabulary (32598, pretrain_t5.py:90) padded to a multiple of 8; enc / dec 512 as BASELINE words it
    "randeng-t5-784m": dict(family="t5", vocab_size=32600, d_model=1024, d_kv=64, d_ff=2816, num_layers=24, num_heads=16,
                            seq=512, seq_dec=512, per_gpu=32, micro=32, lr=1e-4, betas=(0.9, 0.999), wd=0.1, clip=1.0,
                            label="Randeng-T5-784M seq2seq pretrain, enc 512 / dec 512, batch 32/GPU, ZeRO-2 (BASELINE configs[4])"),
    "ziya-llama-13b": dict(family="llama", vocab_size=39424, hidden_size=5120, num_hidden_layers=40,
                           num_attention_heads=40, seq=2048, per_gpu=32, micro=4, lr=1e-4, betas=(0.9, 0.95), wd=0.1,
                           clip=1.0, label="Ziya-LLaMA-13B pretrain, seq 2048, global batch 32/GPU, ZeRO-2 (BASELINE configs[3])"),
}


def workload(name):
    if name in WORKLOADS:
        return dict(WORKLOADS[name])
    if name.startswith("ziya-llama-13b-L"):
        w = dict(WORKLOADS["ziya-llama-13b"])
        w["num_hidden_layers"] = int(name.split("-L")[1])
        w["label"] = f"Ziya-LLaMA-13B WIDTH with {w['num_hidden_layers']} layers (bring-up only, not a BASELINE config)"
        return w
    raise SystemExit(f"unknown workload {name}")


def flops_per_token(w):
    """F_tok = 6*N_mm + 3*F_attn_fwd (causal-counted), SURVEY.md §8(d) / BASELINE.md §3."""
    if w["family"] == "t5":
        from fsb200.models.t5 import t5_flops_per_step
        return t5_flops_per_step(w, 1, w["seq"], w["seq_dec"]) / (w["seq"] + w["seq_dec"])   # per (enc + dec) token
    if w["family"] == "gpt2":
        h, L, V, s = w["n_embd"], w["n_layer"], w["vocab_size"], w["seq"]
        n_mm = L * 12 * h * h + V * h
        attn = 4 * s * h * L / 2
    elif w["family"] == "bert":
        h, L, V, s, ff = w["hidden_size"], w["num_hidden_layers"], w["vocab_size"], w["seq"], w["intermediate_size"]
        n_mm = L * (4 * h * h + 2 * h * ff) + h * h + V * h      # + MLM transform dense + tied decoder
        attn = 4 * s * h * L                                      # bidirectional: full s x s
    else:
        h, L, V, s = w["hidden_size"], w["num_hidden_layers"], w["vocab_size"], w["seq"]
        ff = 256 * ((int(2 * h * 4 / 3) + 255) // 256)
        n_mm = L * (4 * h * h + 3 * h * ff) + V * h
        attn = 4 * s * h * L / 2
    return 6.0 * n_mm + 3.0 * attn


# DRAM traffic of the dominant kernel's largest-share launch: parsed AT RUN TIME from the committed `ncu --set full`
# summaries under profiles/ (dram__bytes_read.sum + dram__bytes_write.sum of ONE launch), next to its algorithmic bytes
# (A + B read once, D written once). Newest round first; null when no committed capture names the shape.
NCU_SHAPES = {
    "gpt2": ("32768x3072x768", "fsb::gemm_bf16_kernel<NN,256,pair> 32768x3072x768 (c_fc forward)", (32768, 3072, 768)),
    "bert": ("32768x3072x768", "fsb::gemm_bf16_kernel<NN,256,pair> 32768x3072x768 (same MLP shape family)", (32768, 3072, 768)),
    "llama": ("8192x15360x5120", "fsb::gemm_bf16_kernel<NT,256,pair> 8192x15360x5120 (QKV forward)", (8192, 15360, 5120)),
    "t5": ("16384x5632x1024", "fsb::gemm_bf16_kernel<NT,256,pair> 16384x5632x1024 (wi_0|wi_1 forward)", (16384, 5632, 1024)),
}
NCU_FILES = ("profiles/r02_ncu_gemm.summary.txt", "profiles/r01_ncu_gemm_final.summary.txt")
_UNIT = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}


def ncu_traffic(family):
    marker, launch, (M, N, K) = NCU_SHAPES.get(family, (None, None, (0, 0, 0)))
    if marker is None:
        return None
    for rel in NCU_FILES:
        path = os.path.join(ROOT, rel)
        if not os.path.exists(path):
            continue
        block, hit = [], False
        for line in open(path):
            if line.startswith("=="):
                if hit:
                    break
                hit = marker in line
                continue
            if hit:
                block.append(line.split())
        if not hit and not block:
            continue
        vals = {t[0]: (float(t[1]), t[2] if len(t) > 2 else "") for t in block if len(t) >= 2}
        try:
            rd = vals["dram__bytes_read.sum"][0] * _UNIT[vals["dram__bytes_read.sum"][1]]
            wr = vals["dram__bytes_write.sum"][0] * _UNIT[vals["dram__bytes_write.sum"][1]]
        except KeyError:
            continue
        tp = vals.get("sm__pipe_tensor_cycles_active.avg.pct_of_peak_sustained_active", (None,))[0]
        return {"launch": launch, "traffic": rd + wr, "dram_read": rd, "dram_write": wr,
                "algorithmic": (M * K + K * N + M * N) * 2.0, "tensor_pipe_active_pct": tp, "source": rel}
    return None


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"bf16_tflops": d.get("bf16_tflops_sustained", d.get("bf16_tflops")), "bf16_burst": d.get("bf16_tflops"),
                "hbm_gbs": d.get("hbm_gbs"), "src": "measured (MEASURED_PEAKS.json, sustained)"}
    return {"bf16_tflops": 1400.0, "bf16_burst": None, "hbm_gbs": 6650.0, "src": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """nvidia-smi clocks/throttle sampling DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms",
                                       "100", "-i", str(gpu_index)], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        if self.p is None:
            return None
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [r.strip().split(",") for r in open(self.f.name) if r.strip()]
        os.unlink(self.f.name)
        sm, mx, reasons = [], [], set()
        for r in rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                if v.strip().lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return None
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


def make_host_batches(w, n_pool, rank):
    """Per-rank synthetic token batches in pinned host memory: g = manual_seed(1234 + dp_rank) (SURVEY.md §8d)."""
    g = torch.Generator().manual_seed(1234 + rank)
    out = []
    for _ in range(n_pool):
        ids = torch.randint(1, w["vocab_size"] - 8, (w["micro"], w["seq"]), generator=g, dtype=torch.int64)
        if w["family"] == "t5":     # span-corruption-shaped: encoder ids, decoder labels (HF shifts them right itself)
            lab = torch.randint(1, w["vocab_size"] - 8, (w["micro"], w["seq_dec"]), generator=g, dtype=torch.int64)
            out.append({"input_ids": ids.pin_memory(), "labels": lab.pin_memory()})
            continue
        if w["family"] == "bert":   # MLM: labels = -100 except a Bernoulli(0.15) subset (SURVEY.md §8d); C3 adds NSP labels
            sel = torch.rand(ids.shape, generator=g) < 0.15
            b = {"input_ids": ids.pin_memory(), "labels": torch.where(sel, ids, torch.full_like(ids, -100)).pin_memory(),
                 "token_type_ids": torch.zeros_like(ids).pin_memory()}
            if w["variant"] == "megatron":
                b["next_sentence_label"] = torch.randint(0, 2, (w["micro"],), generator=g, dtype=torch.int64).pin_memory()
        else:
            b = {"input_ids": ids.pin_memory(), "labels": ids.clone().pin_memory()}
        out.append(b)
    return out


def build_model(w, device, world):
    from types import SimpleNamespace
    if w["family"] == "gpt2":
        from fsb200.models.gpt2 import GPT2LMHeadModel
        cfg = SimpleNamespace(vocab_size=w["vocab_size"], n_positions=w["n_positions"], n_embd=w["n_embd"],
                              n_layer=w["n_layer"], n_head=w["n_head"], layer_norm_epsilon=1e-5, initializer_range=0.02,
                              resid_pdrop=0.0, embd_pdrop=0.0, attn_pdrop=0.0, activation_function="gelu_new")
        return GPT2LMHeadModel(cfg, device=device, world_size=world)
    if w["family"] == "bert":
        from fsb200.models.bert import BertForMaskedLM, MegatronBertForPreTraining
        cfg = SimpleNamespace(vocab_size=w["vocab_size"], hidden_size=w["hidden_size"],
                              num_hidden_layers=w["num_hidden_layers"], num_attention_heads=w["num_attention_heads"],
                              intermediate_size=w["intermediate_size"], hidden_act=w["hidden_act"],
                              max_position_embeddings=512, type_vocab_size=2, layer_norm_eps=1e-12,
                              hidden_dropout_prob=0.0, attention_probs_dropout_prob=0.0, initializer_range=0.02)
        cls = MegatronBertForPreTraining if w["variant"] == "megatron" else BertForMaskedLM
        return cls(cfg, device=device, world_size=world)
    if w["family"] == "t5":
        from fsb200.models.t5 import MT5ForConditionalGeneration
        cfg = SimpleNamespace(vocab_size=w["vocab_size"], d_model=w["d_model"], d_kv=w["d_kv"], d_ff=w["d_ff"],
                              num_layers=w["num_layers"], num_decoder_layers=w["num_layers"], num_heads=w["num_heads"],
                              relative_attention_num_buckets=32, relative_attention_max_distance=128, dropout_rate=0.0,
                              feed_forward_proj="gated-gelu", tie_word_embeddings=True, layer_norm_epsilon=1e-6,
                              pad_token_id=0, decoder_start_token_id=0)
        return MT5ForConditionalGeneration(cfg, device=device, world_size=world)
    from fsb200.models.llama import LlamaForCausalLM
    cfg = SimpleNamespace(vocab_size=w["vocab_size"], hidden_size=w["hidden_size"],
                          num_hidden_layers=w["num_hidden_layers"], num_attention_heads=w["num_attention_heads"],
                          rms_norm_epsilon=1e-6, max_position_embeddings=2048, rotary_emb_base=10000,
                          llama_mlp_multiple_of=256)
    return LlamaForCausalLM(cfg, device=device, world_size=world)


def timed(fn, steps, world):
    """barrier + sync, K steps between CUDA events, sync + barrier; returns max-over-ranks milliseconds."""
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        fn(i)
    e1.record()
    torch.cuda.synchronize()
    ms = torch.tensor([e0.elapsed_time(e1)], device="cuda")
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        dist.barrier()
    return float(ms.item())


def host_threads():
    """Fixed thread count of the CPU arm: the physical cores this process may run on (hyper-thread siblings only slow MKL
    GEMMs down; an auto-calibrated count made the number swing 2.8x between runs in round 1)."""
    avail = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        import psutil
        phys = psutil.cpu_count(logical=False) or avail
    except Exception:
        phys = avail
    return max(1, min(avail, phys))


def cpu_reference_step(w):
    """Build the reference's own CPU implementation of the step for workload `w` (bounded sample: ONE sequence per step).
    Returns (step_fn, tokens_per_call, kind, sample, layer_scale)."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    if w["family"] == "gpt2":
        import hf_oracle as H
        cfg = dict(vocab_size=w["vocab_size"], n_positions=w["n_positions"], n_embd=w["n_embd"], n_layer=w["n_layer"],
                   n_head=w["n_head"])
        model = H.build_gpt2(cfg, bf16_exact=False)
        opt = torch.optim.AdamW(H.wenzhong_param_groups(model.named_parameters(), w["wd"]), lr=w["lr"])
        B, S = 1, w["seq"]
        batch = H.make_lm_batch(w["vocab_size"], B, S)

        def one():
            loss = model(input_ids=batch["input_ids"], labels=batch["labels"]).loss
            opt.zero_grad(set_to_none=True)
            loss.backward()
            opt.step()
        return one, B * S, "reference", f"transformers GPT2LMHeadModel fp32 + torch AdamW, one step = batch {B} x seq {S}", 1.0
    if w["family"] == "bert":
        import hf_oracle as H
        cfg = dict(vocab_size=w["vocab_size"], hidden_size=w["hidden_size"], num_hidden_layers=w["num_hidden_layers"],
                   num_attention_heads=w["num_attention_heads"], intermediate_size=w["intermediate_size"],
                   max_position_embeddings=512, type_vocab_size=2)
        meg = w["variant"] == "megatron"
        model = (H.build_megatron_bert if meg else H.build_bert)(cfg, bf16_exact=False)
        opt = torch.optim.AdamW(H.wenzhong_param_groups(model.named_parameters(), w["wd"]), lr=w["lr"])
        B, S = (1 if meg else 8), w["seq"]
        batch = H.make_mlm_batch(w["vocab_size"], B, S, nsp=meg)

        def one():
            loss = model(**batch).loss
            opt.zero_grad(set_to_none=True)
            loss.backward()
            opt.step()
        return one, B * S, "reference", f"transformers {type(model).__name__} fp32 + torch AdamW, one step = batch {B} x seq {S}", 1.0
    if w["family"] == "t5":
        import hf_oracle as H
        cfg = dict(vocab_size=w["vocab_size"], d_model=w["d_model"], d_kv=w["d_kv"], d_ff=w["d_ff"],
                   num_layers=w["num_layers"], num_decoder_layers=w["num_layers"], num_heads=w["num_heads"],
                   relative_attention_num_buckets=32, relative_attention_max_distance=128)
        model = H.build_mt5(cfg, bf16_exact=False)
        opt = torch.optim.AdamW(H.wenzhong_param_groups(model.named_parameters(), w["wd"]), lr=w["lr"])
        B = 1
        batch = H.make_t5_batch(w["vocab_size"], B, w["seq"], w["seq_dec"])

        def one():
            loss = model(**batch).loss
            opt.zero_grad(set_to_none=True)
            loss.backward()
            opt.step()
        return one, B * (w["seq"] + w["seq_dec"]), "reference", \
            f"transformers MT5ForConditionalGeneration fp32 + torch AdamW, one step = batch {B} x (enc {w['seq']} + dec {w['seq_dec']})", 1.0
    import llama_oracle as O
    Lr = 1  # one full-width layer + head, extrapolated linearly in L (BASELINE.md §2: full size does not fit host RAM)
    V, h, nh = w["vocab_size"], w["hidden_size"], w["num_attention_heads"]
    sd = {k: torch.nn.Parameter(v) for k, v in O.make_weights(V, h, Lr, bf16_exact=False).items()}
    B, S = 1, w["seq"]
    batch = O.make_batch(V, B, S)
    opt = torch.optim.AdamW(O.param_groups(sd.items(), w["wd"]), lr=w["lr"], betas=w["betas"])

    def one():
        loss, _ = O.forward(sd, batch, nh)
        opt.zero_grad(set_to_none=True)
        loss.backward()
        opt.step()
    sample = (f"oracle/llama_oracle.py fp32 (restatement pinned to the unmodified reference), {Lr} of "
              f"{w['num_hidden_layers']} layers at full width + LM head, one step = batch {B} x seq {S}; time x"
              f"{w['num_hidden_layers']} (linear in L; over-counts the head, i.e. flatters the CPU)")
    return one, B * S, "port", sample, float(w["num_hidden_layers"])


def cpu_reference_run(w, steps, warmup, budget_s=None):
    """Time `steps` bounded-sample steps of the CPU arm after `warmup` untimed ones, at a FIXED thread count.
    With budget_s the loop also stops once that much time has been spent (the N=1 line's cpu_baseline leg)."""
    n_thr = host_threads()
    torch.set_num_threads(n_thr)
    one, tok, kind, sample, layer_scale = cpu_reference_step(w)
    for _ in range(max(1, warmup)):
        one()
    t0 = time.time(); n = 0
    while n < steps:
        one(); n += 1
        if budget_s is not None and time.time() - t0 > budget_s:
            break
    dt = (time.time() - t0) / n * layer_scale
    return {"tokens_per_s": tok / dt, "s_per_step": dt, "steps_timed": n, "tokens_per_step": tok, "kind": kind,
            "sample": sample, "cores": n_thr}


DUMP_PARAMS = 8 << 20   # parameter elements written by --dump-outputs (32 MB as float32)


def dump_outputs(out_dir, loss, stepper):
    """What the timed step hands its caller: the step's mean loss and the updated parameters. Models larger than DUMP_PARAMS
    elements are sampled at fixed positions (seed 0), so two builds run with the same arguments write comparable files."""
    stepper.engine.wait_params()
    params = stepper.model.flat.params
    n = params.numel()
    if n > DUMP_PARAMS:
        idx = torch.randint(0, n, (DUMP_PARAMS,), generator=torch.Generator().manual_seed(0)).sort().values
        params = params[idx.to(params.device)]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "loss.npy"), loss.detach().float().cpu().numpy())
    np.save(os.path.join(out_dir, "params.npy"), params.float().cpu().numpy())


def run_workload(name, args, world, rank, device, pg, steps, warmup, want_e2e=True, profile_steps=2, overrides=None,
                 dump_dir=None):
    """Build the model + engine for workload `name`, warm up, time `steps` optimizer steps with the batches resident in
    HBM (`value`), then through the public API from pinned host memory (`e2e`), then `profile_steps` EXTRA steps with CUDA
    events around every GEMM launch (the roofline block) — the timed regions themselves carry no instrumentation.
    With `dump_dir`, rank 0 writes the outputs of the last `value` step there before any further step runs."""
    from fsb200 import lib as L, ops
    from fsb200.schedules import polynomial_lr
    from fsb200.trainer import PretrainStep
    w = workload(name)
    w.update(overrides or {})
    w["micro"] = min(w["micro"], w["per_gpu"])
    ga = w["per_gpu"] // w["micro"]
    tokens_step_gpu = w["per_gpu"] * (w["seq"] + w.get("seq_dec", 0))
    ftok = flops_per_token(w)
    torch.cuda.reset_peak_memory_stats(device)
    model = build_model(w, device, world)
    total_steps = 1000
    stepper = PretrainStep(model, lambda s_: polynomial_lr(s_, w["lr"], 0.01 * total_steps, total_steps, 1e-7), lr=w["lr"],
                           betas=w["betas"], weight_decay=w["wd"], grad_clip=w["clip"], ga_steps=ga, process_group=pg,
                           stage=w.get("stage", 2), comm_sms=args.comm_sms, cuda_graph=bool(args.cuda_graph) and world == 1)
    pool = 2
    host = [make_host_batches(w, ga, rank) for _ in range(pool)]
    dev = [[{k: v.to(device) for k, v in b.items()} for b in hb] for hb in host]
    h2d = sum(t.numel() * t.element_size() for b in host[0] for t in b.values())
    losses = []
    for i in range(warmup):
        losses.append(stepper.step_device(dev[i % pool]))
    torch.cuda.synchronize()

    k0 = L.kernel_launches
    sampler = ClockSampler(device.index) if rank == 0 else None
    ms = timed(lambda i: losses.append(stepper.step_device(dev[i % pool])), steps, world)
    clocks = sampler.stop() if sampler else None
    launches = L.kernel_launches - k0
    if dump_dir and rank == 0:
        dump_outputs(dump_dir, losses[-1], stepper)
    ms_per_step = ms / steps
    value = world * tokens_step_gpu / (ms_per_step / 1000.0)

    e2e = None
    if want_e2e:
        ms2 = timed(lambda i: stepper.step(host[i % pool]), steps, world)
        e2e = {"value": world * tokens_step_gpu / (ms2 / steps / 1000.0), "unit": "tokens/s",
               "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4}

    gsum, prof_ms = {"launches": 0, "ms": 0.0, "work": 0.0}, 0.0
    if stepper.cuda_graph:        # the per-GEMM events of the roofline block need eager launches
        stepper.cuda_graph = False
    if profile_steps:
        prof = ops.KernelProfiler()
        ops.set_profiler(prof)
        prof_ms = timed(lambda i: stepper.step_device(dev[i % pool]), profile_steps, world)
        ops.set_profiler(None)
        gsum = prof.summary().get("gemm_bf16_kernel", gsum)

    if args.breakdown and rank == 0:
        bp = ops.KernelProfiler()
        L.call_profiler = bp
        torch.cuda.synchronize()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for i in range(2):
            stepper.step_device(dev[i % pool])
        ev1.record()
        torch.cuda.synchronize()
        L.call_profiler = None
        tot = ev0.elapsed_time(ev1)
        rows = sorted(bp.summary().items(), key=lambda kv: -kv[1]["ms"])
        acc = sum(v["ms"] for _, v in rows)
        print(f"[breakdown] {name} 2 steps: {tot:.2f} ms wall on the stream; {acc:.2f} ms inside fsb_* calls "
              f"({100 * acc / tot:.1f}%); the rest is torch-native kernels, NCCL and launch gaps", file=sys.stderr)
        for nm, v in rows:
            print(f"[breakdown] {v['ms']:9.3f} ms {100 * v['ms'] / tot:6.2f}%  n={v['launches']:5d}  {nm}", file=sys.stderr)
    elif args.breakdown:
        for i in range(2):
            stepper.step_device(dev[i % pool])

    stepper.engine.wait_params()
    final_loss = float(losses[-1].item())
    first_loss = float(losses[0].item())
    pk = peaks()
    gemm_tf = gsum["work"] / (gsum["ms"] / 1000.0) / 1e12 if gsum["ms"] > 0 else 0.0
    step_tf = value * ftok / world / 1e12
    tr = ncu_traffic(w["family"])
    out = {
        "name": name, "workload": w["label"], "value": value, "ms_per_step": ms_per_step, "e2e": e2e, "launches": launches,
        "clocks": clocks, "final_loss": final_loss, "first_loss": first_loss, "ftok": ftok, "w": w, "ga": ga,
        "roofline": {"bound": "tensor", "kernel": "fsb::gemm_bf16_kernel (tcgen05)", "achieved": gemm_tf,
                     "peak": pk["bf16_tflops"], "unit": "TFLOP/s", "frac": gemm_tf / pk["bf16_tflops"],
                     "frac_of_burst_peak": gemm_tf / pk["bf16_burst"] if pk.get("bf16_burst") else None,
                     "frac_of_spec_2250": gemm_tf / 2250.0,
                     "traffic": tr["traffic"] if tr else None, "traffic_detail": tr, "peak_source": pk["src"],
                     "timing": f"CUDA events around each GEMM launch in {profile_steps} extra steps after the timed region",
                     "launches_per_step": gsum["launches"] / max(1, profile_steps),
                     "kernel_share_of_step": gsum["ms"] / prof_ms if prof_ms > 0 else None,
                     "step_achieved_tflops_per_gpu": step_tf, "step_frac": step_tf / pk["bf16_tflops"],
                     "step_frac_of_burst_peak": step_tf / pk["bf16_burst"] if pk.get("bf16_burst") else None,
                     "step_frac_of_spec_2250": step_tf / 2250.0},
        "memory": dict(stepper.engine.memory_report(), peak_allocated=torch.cuda.max_memory_allocated(device)),
        "comm_bytes_per_step_per_gpu": stepper.engine.comm_bytes // max(1, stepper.engine.step_count),
    }
    del stepper, model, dev, host
    import gc
    gc.collect()
    torch.cuda.empty_cache()
    return out


def parity_block(world, rank, device):
    """Multi-rank correctness, observed inside the driver's own run: a small LLaMA trains 3 steps over `world` ranks
    (ZeRO-2, clipping, bucketed reduce-scatter / all-gather) and the SAME global batch trains on rank 0 alone with
    gradient accumulation; every rank must hold bit-identical parameters after the all-gather, and the two loss curves /
    parameter sets must agree to bf16 reduction-order noise (SURVEY.md Appendix D)."""
    from types import SimpleNamespace
    from fsb200.engine import ZeroEngine
    from fsb200.models.llama import LlamaForCausalLM
    V, h, nl, nh, S, steps, per_rank = 512, 256, 3, 4, 64, 3, 2   # 3 layers: the ZeRO-2 gradient slots rotate
    cfg = SimpleNamespace(vocab_size=V, hidden_size=h, num_hidden_layers=nl, num_attention_heads=nh, rms_norm_epsilon=1e-6,
                          max_position_embeddings=2048, rotary_emb_base=10000, llama_mlp_multiple_of=256)
    solo_groups = [dist.new_group(ranks=[r]) for r in range(world)]   # collective: every rank creates every group

    def batches(step):
        g = torch.Generator().manual_seed(4321 + step)
        return torch.randint(0, V, (world * per_rank, S), generator=g, dtype=torch.int64)

    def train(model, eng, chunks_of):
        losses = []
        for st in range(steps):
            acc = torch.zeros((), device=device)
            mbs = chunks_of(batches(st))
            for mb in mbs:
                out = model(input_ids=mb.to(device), labels=mb.to(device))
                out.loss.backward()
                eng.backward_done()
                acc += out.loss.detach() / len(mbs)
            eng.step()
            losses.append(acc)
        eng.wait_params()
        return torch.stack(losses)

    m_dp = LlamaForCausalLM(cfg, device=device, world_size=world, seed=7)
    e_dp = ZeroEngine(m_dp, lr=1e-3, betas=(0.9, 0.95), weight_decay=0.1, grad_clip=1.0, ga_steps=1, stage=2)
    l_dp = train(m_dp, e_dp, lambda ids: [ids.chunk(world)[rank]])
    dist.all_reduce(l_dp)
    l_dp /= world
    digest = m_dp.flat.params.view(torch.int16).to(torch.int64)
    digest = torch.stack([digest.sum(), (digest * (torch.arange(digest.numel(), device=device) % 8191 + 1)).sum()])
    all_d = [torch.zeros_like(digest) for _ in range(world)]
    dist.all_gather(all_d, digest)
    identical = all(bool(torch.equal(all_d[0], d)) for d in all_d)
    res = {"config": f"LLaMA h{h} L{nl} V{V} s{S}, {steps} steps, global batch {world * per_rank}, ZeRO-2 + clip 1.0",
           "ranks_hold_identical_params": identical}
    if rank == 0:
        m_1 = LlamaForCausalLM(cfg, device=device, world_size=1, seed=7)
        e_1 = ZeroEngine(m_1, lr=1e-3, betas=(0.9, 0.95), weight_decay=0.1, grad_clip=1.0, ga_steps=world, stage=2,
                         process_group=solo_groups[0])
        l_1 = train(m_1, e_1, lambda ids: list(ids.chunk(world)))
        res["loss_curve_dp"] = [float(x) for x in l_dp]
        res["loss_curve_single_rank_ga"] = [float(x) for x in l_1]
        res["max_abs_loss_diff"] = float((l_dp - l_1).abs().max())
        pd, p1 = m_dp.flat.view("llama.layers.0.mlp.w1.weight").float(), m_1.flat.view("llama.layers.0.mlp.w1.weight").float()
        res["param_max_abs_diff_layer0_w1"] = float((pd - p1).abs().max())
        res["ok"] = bool(identical and res["max_abs_loss_diff"] < 5e-3)
    dist.barrier()
    return res


HEADLINE = {8: ("ziya-llama-13b", 3, 1), 4: ("megatronbert-1.3b", 5, 2)}   # gpus -> (workload, timed steps, warm-up)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workload", default="gpt2-110m")
    ap.add_argument("--impl", default="fsb200", choices=["fsb200", "reference"])
    ap.add_argument("--micro-batch", type=int, default=0)
    ap.add_argument("--per-gpu-batch", type=int, default=0, help="override sequences per GPU per step (profiling only)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-headline", action="store_true", help="skip the BASELINE headline config block at --gpus 8 / 4")
    ap.add_argument("--no-parity", action="store_true", help="skip the cross-rank parity block at --gpus > 1")
    ap.add_argument("--comm-sms", type=int, default=int(os.environ.get("FSB_COMM_SMS", "0")),
                    help="SMs the persistent GEMM grids leave to overlapping NCCL kernels (multi-GPU only)")
    ap.add_argument("--cuda-graph", type=int, default=0,
                    help="1: capture the whole optimizer step in a CUDA graph and replay it (single GPU; launch-bound configs)")
    ap.add_argument("--headline-zero-stage", type=int, default=0,
                    help="override the ZeRO stage of the headline block (diagnostic: 1 = reduce once per optimizer step instead of "
                         "once per micro-batch; BASELINE's C4 is stage 2)")
    ap.add_argument("--no-zero1-variant", action="store_true", help="skip the ZeRO-1 variant of the C4 headline block")
    ap.add_argument("--no-graph-block", action="store_true", help="skip the extra CUDA-graph measurement at --gpus 1")
    ap.add_argument("--breakdown", action="store_true",
                    help="after the timed runs, profile 2 more steps with CUDA events around every fsb_* call and print the "
                         "per-entry-point time table to stderr (diagnostic; not part of the JSON line)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the last step's loss and updated parameters (a fixed sample of at most "
                         f"{DUMP_PARAMS} elements) as float32 DIR/loss.npy and DIR/params.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs records the fsb200 step; the reference arm has nothing to write")
    w = workload(args.workload)
    over = {}
    if args.micro_batch:
        over["micro"] = args.micro_batch
    if args.per_gpu_batch:
        over["per_gpu"] = args.per_gpu_batch
        over["label"] = w["label"] + f" [per-GPU batch overridden to {args.per_gpu_batch}: profiling only]"
    w.update(over)
    w["micro"] = min(w["micro"], w["per_gpu"])
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch one rank per GPU, e.g. python -m torch.distributed.run "
                         f"--nnodes=1 --nproc-per-node {args.gpus} --master-addr 127.0.0.1 --master-port 29500 bench.py --gpus {args.gpus}")
    tokens_per_step_gpu = w["per_gpu"] * (w["seq"] + w.get("seq_dec", 0))
    ftok = flops_per_token(w)
    cfg_common = {"workload": w["label"], "name": args.workload, "seq_len": w["seq"], "per_gpu_batch": w["per_gpu"],
                  "global_batch": w["per_gpu"] * max(1, args.gpus), "micro_batch": w["micro"],
                  "grad_accum": w["per_gpu"] // w["micro"], "zero_stage": w.get("stage", 2), "dropout": 0.0,
                  "flops_per_token": ftok, "l2": "working set (weights + activations, GBs) exceeds the 126 MB L2; no flush"}

    if args.impl == "reference":
        if rank != 0:
            return
        r = cpu_reference_run(w, steps=args.steps, warmup=args.warmup)
        v = r["tokens_per_s"]
        line = {"impl": "reference", "metric": "tokens_per_sec", "value": v, "unit": "tokens/s", "n_gpus": args.gpus,
                "steps": r["steps_timed"], "warmup": max(1, args.warmup), "ms_per_step": 1000.0 * r["s_per_step"],
                "tokens_per_step": r["tokens_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic", "config": cfg_common,
                "cpu_baseline": {"value": v, "unit": "tokens/s", "cores": r["cores"], "kind": r["kind"], "sample": r["sample"]},
                "e2e": {"value": v, "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the fsb200 path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    pg = None
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    from fsb200 import lib as L
    L.load()

    warm = max(3, args.warmup)
    main_run = run_workload(args.workload, args, world, rank, device, pg, args.steps, warm, want_e2e=not args.no_e2e,
                            overrides=over, dump_dir=args.dump_outputs)
    graph_block = None
    if world == 1 and not args.cuda_graph and not args.no_graph_block:
        # the same workload with the whole optimizer step captured in ONE CUDA graph and replayed (bit-identical results,
        # tests/test_llama_gpu.py::test_cuda_graph_step_equals_eager_step). Reported beside `value`, which stays on eager
        # launches so that the N = 1 and N > 1 lines of the scaling run measure the same code path.
        args.cuda_graph = 1
        gr = run_workload(args.workload, args, world, rank, device, pg, args.steps, warm, want_e2e=False, profile_steps=0,
                          overrides=over)
        args.cuda_graph = 0
        graph_block = {"tokens_per_s": gr["value"], "ms_per_step": gr["ms_per_step"], "steps": args.steps,
                       "gpu_launches_replayed": gr["launches"], "speedup_vs_eager": gr["value"] / main_run["value"]}
    parity = None
    if world > 1 and not args.no_parity:
        parity = parity_block(world, rank, device)
    headline = None
    if args.gpus in HEADLINE and not args.no_headline and args.workload == "gpt2-110m":
        hname, hsteps, hwarm = HEADLINE[args.gpus]
        hover = {"stage": args.headline_zero_stage} if args.headline_zero_stage else None
        hr = run_workload(hname, args, world, rank, device, pg, hsteps, hwarm, want_e2e=not args.no_e2e, profile_steps=1,
                          overrides=hover)
        headline = {"workload": hr["workload"], "name": hname, "n_gpus": args.gpus, "tokens_per_s": hr["value"],
                    "ms_per_step": hr["ms_per_step"], "steps": hsteps, "warmup": hwarm, "e2e": hr["e2e"],
                    "global_batch": hr["w"]["per_gpu"] * args.gpus, "micro_batch": hr["w"]["micro"], "grad_accum": hr["ga"],
                    "zero_stage": hr["w"].get("stage", 2), "grad_clip": hr["w"]["clip"], "flops_per_token": hr["ftok"],
                    "step_tflops_per_gpu": hr["roofline"]["step_achieved_tflops_per_gpu"],
                    "step_frac_of_sustained_peak": hr["roofline"]["step_frac"],
                    "step_frac_of_burst_peak": hr["roofline"]["step_frac_of_burst_peak"],
                    "step_frac_of_spec_2250": hr["roofline"]["step_frac_of_spec_2250"],
                    "gemm": {k: hr["roofline"][k] for k in ("achieved", "frac", "frac_of_burst_peak", "frac_of_spec_2250",
                                                            "kernel_share_of_step", "launches_per_step")},
                    "clocks": hr["clocks"], "first_loss": hr["first_loss"], "final_loss": hr["final_loss"],
                    "memory_bytes": hr["memory"], "comm_bytes_per_step_per_gpu": hr["comm_bytes_per_step_per_gpu"],
                    "gpu_launches": hr["launches"]}
        if hname == "ziya-llama-13b" and not args.headline_zero_stage and not args.no_zero1_variant:
            # the same model and batch with ZeRO STAGE 1 semantics (full bf16 gradients accumulate locally, ONE reduce-scatter
            # per bucket and optimizer step instead of one per micro-batch): 1/8 of the gradient traffic and no per-micro-batch
            # fp32 shard accumulation. 131 GB peak per GPU — on 180 GB parts gradient sharding is not needed for this model.
            try:   # memory is symmetric across ranks: an out-of-memory here hits every rank at model construction, before any collective
                vr = run_workload(hname, args, world, rank, device, pg, 3, 1, want_e2e=False, profile_steps=0,
                                  overrides={"stage": 1})
                headline["zero1_variant"] = {"tokens_per_s": vr["value"], "ms_per_step": vr["ms_per_step"], "steps": 3, "warmup": 1,
                                             "step_frac_of_sustained_peak": vr["roofline"]["step_frac"],
                                             "final_loss": vr["final_loss"], "clocks": vr["clocks"], "memory_bytes": vr["memory"],
                                             "comm_bytes_per_step_per_gpu": vr["comm_bytes_per_step_per_gpu"]}
            except torch.cuda.OutOfMemoryError as e:
                headline["zero1_variant"] = {"error": f"out of memory: {str(e)[:120]}"}
                torch.cuda.empty_cache()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    line = {"metric": "tokens_per_sec", "value": main_run["value"], "unit": "tokens/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": warm, "ms_per_step": main_run["ms_per_step"], "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic", "config": cfg_common,
            "roofline": main_run["roofline"], "e2e": main_run["e2e"], "gpu_launches": main_run["launches"],
            "clocks": main_run["clocks"], "final_loss": main_run["final_loss"], "memory_bytes": main_run["memory"],
            "comm_bytes_per_step_per_gpu": main_run["comm_bytes_per_step_per_gpu"]}
    if os.environ.get("FSB_ENGINE_SKIP_COLLECTIVES", "0") == "1":
        line["INVALID_diagnostic"] = ("FSB_ENGINE_SKIP_COLLECTIVES=1: the NCCL calls were dropped (results are wrong); this line only "
                                      "measures the step WITHOUT communication — subtract from the normal run to get the exposed comm")
    if graph_block is not None:
        line["cuda_graph_step"] = graph_block
    if parity is not None:
        line["parity"] = parity
    if headline is not None:
        line["headline"] = headline
    if args.gpus == 1 and not args.no_cpu_baseline:
        r = cpu_reference_run(w, steps=8, warmup=1, budget_s=15.0)
        line["cpu_baseline"] = {"value": r["tokens_per_s"], "unit": "tokens/s", "cores": r["cores"], "kind": r["kind"],
                                "sample": r["sample"]}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
