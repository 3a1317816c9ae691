#!/usr/bin/env python
"""bench.py — audio-seconds/second of one SLAM-LLM LoRA training step (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # this repo's sm_100a step
    python bench.py --impl reference --gpus N --steps K --warmup W   # CPU restatement of the reference path

Workload (config.workload): Whisper-large-v3 + Llama-3-8B, LoRA r=16 on q_proj/v_proj, concat-linear projector (k=5),
4 x 30 s synthetic 16 kHz utterances per GPU (120 audio-s per step per GPU, S = 300 audio + 24 prompt + 77 answer tokens),
random-init weights, fwd + bwd + gradient all-reduce (N>1) + AdamW.  Weak scaling: per-GPU batch fixed.

One JSON line on rank 0:
  value      whole-job audio-s/s with the batch already resident in HBM (device-timed, max over ranks)
  e2e        the same step driven through the public host API from PINNED HOST buffers (H2D of PCM/ids/masks and a
             D2H read of the loss inside the timed region)
  roofline   tcgen05 GEMM family: algorithmic FLOPs / CUDA-event time of every GEMM launch inside the timed steps,
             vs the measured sustained bf16 peak (MEASURED_PEAKS.json)
  cpu_baseline  the oracle (CPU port of the reference path) on the host cores, bounded sample, extrapolated by layer count
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

METRIC = "audio_sec_per_sec"
UNIT = "audio-s/s"
WORKLOADS = {
    "c3": dict(enc="large-v3", llm="llama-3-8b", r=16, alpha=32, targets=("q_proj", "v_proj"), batch=4, seconds=30, prompt=24, answer=76,
               name="whisper-large-v3+llama-3-8b lora(r=16,q/v) linear-proj k=5, 4x30s utt per GPU (120 audio-s/step/GPU), S=401"),
    "c2": dict(enc="base", llm="llama-3-8b", r=16, alpha=32, targets=("q_proj", "v_proj"), batch=4, seconds=30, prompt=24, answer=76,
               name="whisper-base+llama-3-8b lora(r=16,q/v) linear-proj k=5, 4x30s utt per GPU (120 audio-s/step/GPU), S=401"),
    # BASELINE configs[2] batching: utterances U[10 s, 30 s] grouped by the reference's window rule (speech_dataset_large.py:259-263,
    # train_max_frame_length tokens per batch), natural lengths, right padding; value counts REAL audio seconds
    "c3-dynamic": dict(enc="large-v3", llm="llama-3-8b", r=16, alpha=32, targets=("q_proj", "v_proj"), batch=None, seconds=(10, 30), prompt=24, answer=76,
                       max_frame_length=1500, n_batches=8,
                       name="whisper-large-v3+llama-3-8b lora(r=16,q/v) linear-proj k=5, dynamic-frame batches (utt U[10,30] s, window rule 1500 tokens)"),
    "tiny": dict(enc="tiny", llm="tinyllama-1.1b", r=8, alpha=32, targets=("q_proj", "v_proj"), batch=1, seconds=30, prompt=24, answer=76,
                 name="whisper-tiny+tinyllama-1.1b lora(r=8,q/v), 1x30s"),
}


def dist_env():
    return int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))


def make_batch(wl, vocab, seed, pin=False):
    """Synthetic batch in the collator contract (speech_dataset.py:216-291): [audio(-1)*300, prompt, answer, eos]."""
    g = torch.Generator().manual_seed(seed)
    B, n = wl["batch"], wl["seconds"] * 16000
    Ta = ((n // 160 + 1) // 2) // 5
    S = Ta + wl["prompt"] + wl["answer"] + 1
    ids = torch.randint(0, vocab, (B, S), generator=g)
    ids[:, :Ta] = -1
    labels = torch.full((B, S), -100, dtype=torch.int64)
    labels[:, Ta + wl["prompt"]:] = ids[:, Ta + wl["prompt"]:]
    batch = dict(input_ids=ids, labels=labels, attention_mask=torch.ones(B, S, dtype=torch.bool), modality_mask=ids == -1,
                 audio_pcm=torch.randn(B, n, generator=g) * 0.1)
    if pin:
        batch = {k: v.pin_memory() for k, v in batch.items()}
    return batch, S


def make_dynamic_batches(wl, vocab, seed, pin=False):
    """Synthetic stream of natural-length utterances grouped by the reference window rule; right-padding collator contract of
    speech_dataset_large.py:180-233 (audio first, no left padding) with raw PCM + per-utterance lengths (GPU front end)."""
    g = torch.Generator().manual_seed(seed)
    lo, hi = wl["seconds"]
    batches, buf = [], []

    def tokens(n):
        return ((n // 160 + 1) // 2) // 5 + wl["prompt"] + wl["answer"] + 1

    def flush(items):
        B = len(items)
        S = max(tokens(n) for n in items)
        width = max(items)
        ids = torch.zeros(B, S, dtype=torch.int64)
        labels = torch.full((B, S), -100, dtype=torch.int64)
        att = torch.zeros(B, S, dtype=torch.bool)
        mod = torch.zeros(B, S, dtype=torch.bool)
        pcm = torch.zeros(B, width)
        for b, n in enumerate(items):
            ta = ((n // 160 + 1) // 2) // 5
            nt = tokens(n)
            ids[b, ta:nt] = torch.randint(0, vocab, (nt - ta,), generator=g)
            ids[b, :ta] = -1
            labels[b, ta + wl["prompt"]:nt] = ids[b, ta + wl["prompt"]:nt]
            att[b, :nt] = True
            mod[b, :ta] = True
            pcm[b, :n] = torch.randn(n, generator=g) * 0.1
        batch = dict(input_ids=ids, labels=labels, attention_mask=att, modality_mask=mod, audio_pcm=pcm,
                     audio_pcm_lengths=torch.tensor(items, dtype=torch.int32))
        if pin:
            batch = {k: v.pin_memory() for k, v in batch.items()}
        return batch, sum(items) / 16000.0, B * width / 16000.0

    while len(batches) < wl["n_batches"]:
        n = int(torch.randint(lo * 16000, hi * 16000 + 1, (1,), generator=g))
        longest = max([tokens(n)] + [tokens(m) for m in buf])
        if buf and (len(buf) + 1) * longest > wl["max_frame_length"]:
            batches.append(flush(buf))
            buf = []
        buf.append(n)
    return batches


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc, self.t_mark = index, [], None, 0.0

    def mark(self):
        """Start of the timed region: only samples that arrive after this call are reported (the sampler itself is started before the
        warm-up so that short timed regions still see several 100 ms samples)."""
        self.t_mark = time.perf_counter()

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [x.strip() for x in line.split(",")]))

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        self.rows = [r for t, r in self.rows if t >= self.t_mark]
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for j, n in enumerate(names) if any(len(r) > 3 + j and r[3 + j].lower().startswith("active") for r in self.rows)]
        pw = [float(r[2]) for r in self.rows if len(r) > 2 and r[2].replace(".", "").isdigit()]
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "power_w_max": max(pw) if pw else None, "samples": len(sm)}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("bf16_tflops_sustained", 1467.7), d.get("hbm_gbs", 6570.6), "measured (MEASURED_PEAKS.json, sustained)"
    return 1400.0, 6650.0, "fallback (B200_PROFILING.md)"


# ----------------------------------------------------------------------------------------------------------------------
# CPU baseline: the oracle (port of the reference's eager path) on the host cores, bounded sample
# ----------------------------------------------------------------------------------------------------------------------
def pick_cpu_threads():
    """Use as many host threads as actually help: the box may expose more logical CPUs than its cgroup quota grants, in
    which case torch with os.cpu_count() threads is several times SLOWER.  Time one decoder-MLP-shaped matmul at a few
    thread counts and keep the fastest (the count is reported as cpu_baseline.cores)."""
    try:
        avail = len(os.sched_getaffinity(0))
    except AttributeError:
        avail = os.cpu_count() or 1
    cands = sorted({c for c in (avail, avail // 2, 64, 32, 16, 8) if 1 <= c <= avail}, reverse=True)
    a, b = torch.randn(401, 4096), torch.randn(4096, 14336)
    best, best_t = cands[-1], float("inf")
    for c in cands:
        torch.set_num_threads(c)
        torch.mm(a, b)
        t0 = time.perf_counter()
        for _ in range(3):
            torch.mm(a, b)
        t = time.perf_counter() - t0
        if t < best_t * 0.95:
            best, best_t = c, t
    torch.set_num_threads(best)
    return best


def cpu_reference(wl, steps, warmup, budget_s=150.0, quiet=True):
    """Times the CPU restatement of the reference path (oracle/slam_oracle.py) on one utterance with a reduced number of
    encoder/decoder layers and extrapolates linearly in the layer counts to the full depth.  Returns audio-s/s."""
    from oracle import slam_oracle as so
    cores = pick_cpu_threads()
    enc_full, llm_full = so.WHISPER[wl["enc"]], so.LLM[wl["llm"]]
    lora, proj = so.LoraCfg(wl["r"], wl["alpha"], tuple(wl["targets"])), so.ProjCfg("linear", 5, 2048)
    wl1 = dict(wl, batch=1)
    batch, S = make_batch(wl1, llm_full.vocab, seed=42)

    def build(n_enc, n_dec):
        enc = so.EncoderCfg(enc_full.n_mels, enc_full.n_ctx, enc_full.d, enc_full.heads, n_enc)
        llm = so.LlmCfg(llm_full.vocab, llm_full.d, n_dec, llm_full.heads, llm_full.kv_heads, llm_full.ffn, llm_full.rope_theta, llm_full.eps)
        g = torch.Generator().manual_seed(1)

        def n(*s):
            return torch.empty(*s).normal_(0, 0.02, generator=g)
        ew = {"conv1.weight": n(enc.d, enc.n_mels, 3), "conv1.bias": n(enc.d), "conv2.weight": n(enc.d, enc.d, 3), "conv2.bias": n(enc.d),
              "positional_embedding": so.sinusoids(enc.n_ctx, enc.d), "ln_post.weight": torch.ones(enc.d), "ln_post.bias": torch.zeros(enc.d)}
        for i in range(n_enc):
            p = f"blocks.{i}."
            ew.update({p + "attn.query.weight": n(enc.d, enc.d), p + "attn.query.bias": n(enc.d), p + "attn.key.weight": n(enc.d, enc.d),
                       p + "attn.value.weight": n(enc.d, enc.d), p + "attn.value.bias": n(enc.d), p + "attn.out.weight": n(enc.d, enc.d),
                       p + "attn.out.bias": n(enc.d), p + "attn_ln.weight": torch.ones(enc.d), p + "attn_ln.bias": torch.zeros(enc.d),
                       p + "mlp.0.weight": n(4 * enc.d, enc.d), p + "mlp.0.bias": n(4 * enc.d), p + "mlp.2.weight": n(enc.d, 4 * enc.d),
                       p + "mlp.2.bias": n(enc.d), p + "mlp_ln.weight": torch.ones(enc.d), p + "mlp_ln.bias": torch.zeros(enc.d)})
        lw = {"model.embed_tokens.weight": n(llm.vocab, llm.d), "model.norm.weight": torch.ones(llm.d), "lm_head.weight": n(llm.vocab, llm.d)}
        for i in range(n_dec):
            p = f"model.layers.{i}."
            for nm in ("q_proj", "k_proj", "v_proj", "o_proj"):
                lw[p + f"self_attn.{nm}.weight"] = n(*so.linear_shape(llm, nm))
            for nm in ("gate_proj", "up_proj", "down_proj"):
                lw[p + f"mlp.{nm}.weight"] = n(*so.linear_shape(llm, nm))
            lw[p + "input_layernorm.weight"] = torch.ones(llm.d)
            lw[p + "post_attention_layernorm.weight"] = torch.ones(llm.d)
        return so.OracleModel(enc, llm, lora, proj, ew, lw, so.init_lora(llm, lora, 2), so.init_projector(enc, llm, proj, 3))

    def timed_step(model):
        t0 = time.perf_counter()
        model.step(dict(batch), lr=1e-4)
        return time.perf_counter() - t0

    m0 = build(0, 0)
    timed_step(m0)
    t_fixed = min(timed_step(m0) for _ in range(2))            # front end + conv stem + projector + merge + lm_head/CE + their backward
    del m0
    per_step_budget = max(2.0, budget_s / max(1, steps + warmup))
    m1 = build(1, 1)
    timed_step(m1)
    t_one = timed_step(m1)
    per_layer = max(t_one - t_fixed, 1e-3)
    n_lay = int(max(1, min(8, (per_step_budget - t_fixed) // per_layer)))
    if n_lay != 1:
        del m1
        m1 = build(min(n_lay, enc_full.layers), min(n_lay, llm_full.layers))
    n_enc, n_dec = m1.enc_cfg.layers, m1.llm_cfg.layers
    for _ in range(warmup):
        timed_step(m1)
    ts = [timed_step(m1) for _ in range(steps)]
    t_sample = sum(ts) / len(ts)
    # encoder layer share measured once (no-grad forward of the sample's encoder), the rest is decoder fwd+bwd
    mel = so.batch_log_mel(batch["audio_pcm"], enc_full.n_mels)
    t0 = time.perf_counter()
    with torch.no_grad():
        so.whisper_encoder(m1.enc_w, m1.enc_cfg, mel)
    t_enc_n = time.perf_counter() - t0
    m1.enc_cfg.layers, saved = 0, m1.enc_cfg.layers
    t0 = time.perf_counter()
    with torch.no_grad():
        so.whisper_encoder(m1.enc_w, m1.enc_cfg, mel)
    t_enc_0 = time.perf_counter() - t0
    m1.enc_cfg.layers = saved
    t_enc_layer = max(t_enc_n - t_enc_0, 0.0) / max(n_enc, 1)
    t_dec_layer = max(t_sample - t_fixed - n_enc * t_enc_layer, 1e-3) / n_dec
    t_full_utt = t_fixed + enc_full.layers * t_enc_layer + llm_full.layers * t_dec_layer
    value = wl["seconds"] / t_full_utt                           # audio-s/s, batch scales linearly on a CPU
    sample = (f"B=1 x {wl['seconds']} s utterance, {n_enc}/{enc_full.layers} encoder + {n_dec}/{llm_full.layers} decoder layers, fp32, "
              f"{steps} timed steps of {t_sample:.2f} s; extrapolated linearly in layer count to full depth "
              f"(fixed {t_fixed:.2f} s + {enc_full.layers}x{t_enc_layer:.3f} s + {llm_full.layers}x{t_dec_layer:.3f} s per utterance)")
    return dict(value=value, unit=UNIT, cores=cores, kind="port", sample=sample), t_sample


# ----------------------------------------------------------------------------------------------------------------------
# the recipe surface: model built by setup_encoder / setup_llm / setup_encoder_projector + slam_model, driven by train()
# ----------------------------------------------------------------------------------------------------------------------
def build_recipe_model(wl, enc, llm, lora, world):
    """What a recipe's model_factory does (examples/asr_librispeech/model/slam_model_asr.py:15-55) minus the tokenizer download: a config.json
    of the LLM architecture in a temp dir, `b200_random_init` for the frozen weights (no checkpoints offline), LoRA B ~ N(0, 0.02) so that
    dA != 0 (peft would zero-init B)."""
    import tempfile
    sys.path.insert(0, os.path.join(ROOT, "src"))
    import slam_llm  # noqa: F401  (installs the omegaconf / hydra / whisper shims when the real packages are absent)
    from omegaconf import OmegaConf
    from slam_llm.models.slam_model import setup_encoder, setup_encoder_projector, setup_llm, slam_model
    tmp = tempfile.mkdtemp(prefix="slam_bench_llm_")
    json.dump(dict(model_type="llama", vocab_size=llm.vocab, hidden_size=llm.d, intermediate_size=llm.ffn, num_hidden_layers=llm.layers,
                   num_attention_heads=llm.heads, num_key_value_heads=llm.kv_heads, rms_norm_eps=llm.eps, rope_theta=llm.rope_theta),
              open(os.path.join(tmp, "config.json"), "w"))
    train_config = OmegaConf.create(dict(
        model_name="bench", enable_fsdp=False, enable_ddp=False, enable_deepspeed=False, quantization=False, freeze_llm=True, freeze_encoder=True,
        use_peft=True, seed=42, num_epochs=1, batching_strategy="custom", gradient_accumulation_steps=1, run_validation=False, validation_interval=10 ** 9,
        save_model=False, use_fp16=False, lr=1e-4, weight_decay=0.0, warmup_steps=1000, total_steps=100000, output_dir=tmp,
        peft_config=dict(peft_method="lora", r=lora.r, lora_alpha=lora.alpha, target_modules=list(lora.targets), bias="none", task_type="CAUSAL_LM",
                         lora_dropout=0.0, inference_mode=False)))
    model_config = OmegaConf.create(dict(llm_name=wl["llm"], llm_path=tmp, llm_dim=llm.d, encoder_name="whisper", encoder_path=wl["enc"], encoder_dim=enc.d,
                                         encoder_projector="linear", encoder_projector_ds_rate=5, b200_random_init=True))
    torch.cuda.manual_seed(train_config.seed)                      # as finetune.main does: the projector's nn.Linear init draws from the global RNG
    torch.manual_seed(train_config.seed)
    encoder = setup_encoder(train_config, model_config)
    llm_mod = setup_llm(train_config, model_config)
    projector = setup_encoder_projector(train_config, model_config)
    model = slam_model(encoder, llm_mod, projector, None, train_config, model_config, metric="acc")
    with torch.no_grad():
        model.b200.llm.init_lora(None, seed=44, b_std=0.02)
    return model, train_config


class _SyntheticUtterances(torch.utils.data.Dataset):
    """Map-style dataset of synthetic utterances in the item layout of datasets/speech_dataset.py:109-161 ([audio(-1)*L, prompt, answer, eos]),
    a fresh waveform per item; batches are formed by the repo's SpeechDatasetJsonl.collator (the reference collator contract)."""

    def __init__(self, wl, vocab, n_items, seed):
        from slam_llm.datasets.speech_dataset import SpeechDatasetJsonl
        self.wl, self.vocab, self.n, self.seed = wl, vocab, n_items, seed
        c = SpeechDatasetJsonl.__new__(SpeechDatasetJsonl)
        c.tokenizer = type("Tok", (), {"pad_token_id": 0, "eos_token_id": 2})()
        c.input_type, c.inference_mode = "mel", False
        self._collator = c

    def __len__(self):
        return self.n

    def __getitem__(self, i):
        g = torch.Generator().manual_seed(self.seed * 100003 + i)
        n = self.wl["seconds"] * 16000
        ta = ((n // 160 + 1) // 2) // 5
        text = torch.randint(3, self.vocab, (self.wl["prompt"] + self.wl["answer"] + 1,), generator=g)
        ids = torch.cat((torch.full((ta,), -1), text))
        labels = ids.clone()
        labels[: ta + self.wl["prompt"]] = -100
        att = ids.ge(-1)
        return dict(input_ids=ids, labels=labels, attention_mask=att, audio=None, audio_mel=None, audio_pcm=torch.randn(n, generator=g) * 0.1,
                    audio_length=ta, prompt_length=self.wl["prompt"])

    def collator(self, samples):
        return self._collator.collator(samples)


def recipe_leg(wl, model, train_config, llm, audio_s, steps, warmup, rank=0, local_rank=0, world=1):
    """`e2e_recipe`: slam_llm.utils.train_utils.train() (the reference's loop, utils/train_utils.py:46-392) over a DataLoader (2 workers, pinned
    memory) of FRESH synthetic batches: collate, H2D, label rows, model(**batch), outputs.loss.backward(), FlatAdamW.step(), LambdaLR.step(), the
    per-step tqdm description (one D2H read per step).  Wall-clock around the whole epoch of `steps` batches, device synchronised on both sides."""
    from omegaconf import OmegaConf
    from slam_llm.utils.train_utils import train
    from slam_llm_b200.optim import FlatAdamW
    log_config = OmegaConf.create(dict(use_wandb=False, log_interval=10))
    if world > 1:                                                  # what pipeline/finetune.py sets up for enable_ddp (finetune.py:84-90 of the mirror)
        train_config.enable_ddp = True
        model.ddp_world_size = world
        model.b200.defer_update = True
    optimizer = FlatAdamW(model, lr=train_config.lr, weight_decay=train_config.weight_decay)
    scheduler = torch.optim.lr_scheduler.LambdaLR(optimizer, lr_lambda=lambda step: min((step + 1) / train_config.warmup_steps, 1))

    ds = _SyntheticUtterances(wl, llm.vocab, steps * wl["batch"], seed=2 + rank)
    dl = torch.utils.data.DataLoader(ds, batch_size=wl["batch"], num_workers=2, pin_memory=True, collate_fn=ds.collator, drop_last=True,
                                     persistent_workers=True, prefetch_factor=4)

    class _Stamped:
        """The DataLoader with a time stamp at every batch hand-over (train() reads the loss on the host every step, so the stamps are
        step boundaries): separates the steady state from the per-epoch fixed cost (MemoryTrace's empty_cache -> the first steps re-grow
        the caching allocator with cudaMalloc; irrelevant for real epochs of thousands of steps, dominant for a 20-step one)."""

        def __init__(self, loader):
            self.loader, self.stamps = loader, []

        def __len__(self):
            return len(self.loader)

        def __iter__(self):
            for b in self.loader:
                self.stamps.append(time.perf_counter())
                yield b

    def epoch():
        st = _Stamped(dl)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        res = train(model, st, None, None, optimizer, scheduler, 1, train_config, log_config, None, local_rank if world > 1 else None,
                    rank if world > 1 else None)
        model.b200.flush_update()
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        skip = min(4, steps // 2)                                 # hand-over to hand-over: excludes the epoch's enter/exit work
        steady = (st.stamps[-1] - st.stamps[skip]) / max(len(st.stamps) - 1 - skip, 1)
        return t1 - t0, steady, res

    t_first, _, _ = epoch()                                       # warm-up epoch: also pays the DataLoader worker start-up (fork + first prefetch)
    t, steady, res = epoch()                                      # timed epoch: the same persistent workers, `steps` fresh batches
    del dl
    if world > 1:                                                 # slowest rank decides
        tt = torch.tensor([steady, t], device=model.b200.device, dtype=torch.float64)
        torch.distributed.all_reduce(tt, op=torch.distributed.ReduceOp.MAX)
        steady, t = float(tt[0]), float(tt[1])
        train_config.enable_ddp = False
    ms = steady * 1e3
    return {"value": round(world * audio_s / (ms / 1e3), 2), "unit": UNIT, "ms_per_step": round(ms, 3), "steps": steps,
            "whole_epoch_ms_per_step": round(t * 1e3 / steps, 3), "first_epoch_ms_per_step": round(t_first * 1e3 / steps, 3),
            "measured": "steady state of the timed epoch: wall clock from the hand-over of batch 5 to the hand-over of batch K (train() reads the loss "
                        "on the host every step, so hand-overs are step boundaries); whole_epoch also pays MemoryTrace's per-epoch gc + empty_cache "
                        "(cudaFree / cudaMalloc re-growth of ~8 GB of activations) amortised over only K steps",
            "path": "slam_llm.utils.train_utils.train() + DataLoader(2 persistent workers, fresh batch per step, collator, pinned H2D, label rows) + "
                    "model(**batch) + loss.backward() + FlatAdamW + LambdaLR + per-step tqdm loss read; wall clock of one epoch after a warm-up epoch",
            "avg_train_loss": round(float(res["avg_train_loss"]), 4)}


# ----------------------------------------------------------------------------------------------------------------------
# B-EAGER: the reference's eager HF/PEFT step on the same GPU, same batch (baseline/eager_hf.py); N=1 only
# ----------------------------------------------------------------------------------------------------------------------
def eager_baseline(wl, enc, llm, lora, host_batch, dev, eng, audio_s, our_e2e, steps=20, warmup=5, model=None):
    """Frees this repo's engine state, builds HF WhisperEncoder + LlamaForCausalLM (fp32 master weights) with restated peft LoRA, and times the
    reference train-loop body (fp16 autocast + GradScaler + AdamW, train_utils.py:112-149) on the same synthetic batch; the log-mel the
    reference computes in its DataLoader workers is prepared outside the timed region (generous to the baseline)."""
    try:
        from baseline import eager_hf
        mel = eng.log_mel(host_batch["audio_pcm"].to(dev)).float().cpu()
        for k in list(vars(eng)):                                   # drop every device tensor the step owns (the recipe modules only hold views)
            setattr(eng, k, None)
        if model is not None:
            model.encoder.b200 = model.llm.b200 = model.b200 = None
        import gc
        gc.collect()
        torch.cuda.empty_cache()
        r = eager_hf.run(enc, llm, lora, host_batch, mel, steps=steps, warmup=warmup, device=dev)
        value = audio_s / (r["ms_per_step"] / 1e3)
        return {"value": round(value, 2), "unit": UNIT, "ms_per_step": round(r["ms_per_step"], 2), "wall_ms_per_step": round(r["wall_ms_per_step"], 2),
                "steps": steps, "warmup": warmup, "dtype": "fp16 autocast over fp32 master weights + GradScaler", "same_config": True,
                "path": "HF WhisperEncoder modules (sdpa) + HF LlamaForCausalLM (eager attention) + restated peft-0.6 LoRA + torch.optim.AdamW; "
                        "batch incl. CPU-side log-mel resident on the device", "peak_mem_gb": r["peak_mem_gb"],
                "speedup_e2e": round(our_e2e / value, 2), "last": r["last"]}
    except Exception as e:  # the baseline leg must never take the bench line down
        return {"unavailable": f"{type(e).__name__}: {e}"[:300]}


# ----------------------------------------------------------------------------------------------------------------------
# N>1 diagnostic: where does the weak-scaling loss come from?
# ----------------------------------------------------------------------------------------------------------------------
def scale_breakdown(args, eng, dev_batch, lr, rank, world, dev, steps=20):
    """Per-rank device time of `steps` steps in three modes: (a) independent replicas (no collective: pure per-GPU speed under the shared
    power/thermal envelope), (b) blocking all-reduce after backward (round-1 design), (c) async all-reduce + deferred AdamW.  Also the host
    enqueue time per step and, for (b), the device time spent inside the all-reduce (which includes waiting for the slowest rank)."""
    import torch.distributed as dist
    if world == 1:
        class dist:  # noqa: N801  (single process: no collectives)
            barrier = staticmethod(lambda: None)
            all_gather_object = staticmethod(lambda out, obj: out.__setitem__(0, obj))

    def run(mode):
        eng.flush_update()
        eng.defer_update = mode == "overlap"
        ar_events = []
        for it in range(3 + steps):
            if it == 3:
                dist.barrier()
                torch.cuda.synchronize()
                t_host = time.perf_counter()
                e0 = torch.cuda.Event(enable_timing=True)
                e0.record()
            loss, acc, _ = eng.forward(dev_batch, train=True)
            eng.backward()
            if mode == "blocking":
                a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a0.record()
                eng.allreduce_grads(async_op=False)
                a1.record()
                if it >= 3:
                    ar_events.append((a0, a1))
            elif mode == "overlap":
                eng.allreduce_grads(async_op=True)
            eng.optimizer_step(lr, 0.0, grad_div=float(world) if mode != "independent" else 1.0)
        eng.flush_update()
        e1 = torch.cuda.Event(enable_timing=True)
        e1.record()
        host_ms = (time.perf_counter() - t_host) * 1e3 / steps
        torch.cuda.synchronize()
        out = {"ms_per_step": e0.elapsed_time(e1) / steps, "host_enqueue_ms_per_step": host_ms}
        if ar_events:
            out["allreduce_ms_per_step"] = sum(a.elapsed_time(b) for a, b in ar_events) / len(ar_events)
        return out

    def host_only():
        """Pure host cost of enqueueing one step: device idle and launch queue empty at the start, no synchronisation inside."""
        eng.flush_update()
        eng.defer_update = False
        ts = []
        for _ in range(4):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            eng.forward(dev_batch, train=True)
            t1 = time.perf_counter()
            eng.backward()
            t2 = time.perf_counter()
            eng.optimizer_step(lr, 0.0)
            t3 = time.perf_counter()
            ts.append((t1 - t0, t2 - t1, t3 - t2))
        torch.cuda.synchronize()
        best = min(ts, key=sum)
        return {"forward_ms": best[0] * 1e3, "backward_ms": best[1] * 1e3, "optimizer_ms": best[2] * 1e3, "total_ms": sum(best) * 1e3}

    modes = ("independent", "blocking", "overlap") if world > 1 else ("independent",)
    res = {m: run(m) for m in modes}
    res["host_only"] = host_only()
    try:
        smi = subprocess.run(["nvidia-smi", f"--id={dev.index}", "--query-gpu=clocks.sm,power.draw,temperature.gpu", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=10).stdout.strip()
    except Exception:
        smi = ""
    res["smi_after"] = smi
    gathered = [None] * world
    dist.all_gather_object(gathered, res)
    if rank == 0:
        summary = {m: {"max_ms": max(g[m]["ms_per_step"] for g in gathered), "min_ms": min(g[m]["ms_per_step"] for g in gathered)} for m in modes}
        summary["host_only_total_ms"] = {"max": max(g["host_only"]["total_ms"] for g in gathered), "min": min(g["host_only"]["total_ms"] for g in gathered)}
        os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
        with open(os.path.join(ROOT, "gpurun_out", f"scale_breakdown_n{world}.json"), "w") as f:
            json.dump({"world": world, "steps": steps, "summary": summary, "ranks": gathered}, f, indent=1)
        print("[breakdown] " + json.dumps(summary), file=sys.stderr, flush=True)
    eng.defer_update = world > 1 and args.overlap == 1


# ----------------------------------------------------------------------------------------------------------------------
def parse_gemm_traffic(log):
    """ncu `--csv --log-file` output -> {launch id: DRAM bytes read + written} for the GEMM kernels of this library."""
    import csv
    scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    per = {}
    for row in csv.DictReader(l for l in open(log) if not l.startswith("==")):
        name = row.get("Kernel Name", "")
        if "gemm_tcgen05" not in name and "gemm_thin_cluster" not in name:
            continue
        try:
            per[row["ID"]] = per.get(row["ID"], 0.0) + float(row["Metric Value"].replace(",", "")) * scale.get(row["Metric Unit"], 1.0)
        except (KeyError, ValueError):
            continue
    return per


def measure_gemm_traffic(workload, budget_s=240.0):
    """roofline.traffic measured in THIS run: one eager step of the same workload in a child process under `ncu`
    (dram__bytes_read.sum + dram__bytes_write.sum of every GEMM launch, per launch).  Hardware counters cannot be read from inside the
    timed process, so the child rebuilds the same step (same code, same shapes, same box); returns (bytes per launch | None, how)."""
    import shutil
    import subprocess
    import tempfile
    ncu = shutil.which("ncu") or "/usr/local/cuda/bin/ncu"
    if not os.path.exists(ncu):
        return None, "ncu not found"
    with tempfile.TemporaryDirectory() as td:
        log = os.path.join(td, "gemm_traffic.csv")
        cmd = [ncu, "--profile-from-start", "off", "--metrics", "dram__bytes_read.sum,dram__bytes_write.sum", "--clock-control", "none", "--csv",
               "--log-file", log, sys.executable, os.path.abspath(__file__), "--ncu-step", "--graph", "0", "--skip-cpu", "--skip-eager", "--skip-recipe",
               "--skip-traffic", "--workload", workload]
        env = {k: v for k, v in os.environ.items() if k not in ("RANK", "LOCAL_RANK", "WORLD_SIZE", "MASTER_ADDR", "MASTER_PORT")}
        try:
            r = subprocess.run(cmd, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL, timeout=budget_s, env=env)
        except subprocess.TimeoutExpired:
            return None, f"ncu child exceeded {budget_s:.0f} s"
        if not os.path.exists(log):
            return None, f"ncu child wrote no log (rc={r.returncode})"
        per = parse_gemm_traffic(log)
    if not per:
        return None, "no GEMM launches in the ncu log"
    return round(sum(per.values()) / len(per)), f"measured in this run: ncu child process, one eager step of the same workload, {len(per)} GEMM launches"


def dump_outputs(out_dir, loss, acc, eng, sample=1 << 22):
    """What the last timed step hands its caller, as float32 .npy files: the loss and the token accuracy it returns, and the trainable
    parameters after its AdamW update (every trainable, concatenated in name order, at 4M fixed seeded positions: 16 MB).
    Some gradient reductions use atomics, so two runs agree only up to rounding that the steps amplify (B200, 1000 W, 3 warm-up +
    10 timed steps, two pairs of runs: loss within 1.3e-3, parameters within 6e-3 relative L2)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    state = eng.trainable_state("param")
    params = torch.cat([state[k].detach().float().reshape(-1) for k in sorted(state)])
    if params.numel() > sample:
        idx = torch.randperm(params.numel(), generator=torch.Generator().manual_seed(0))[:sample].sort().values
        params = params[idx.to(params.device)]
    arrays = {"loss": loss.detach().float().reshape(1), "accuracy": acc.detach().float().reshape(1), "trainable_params": params}
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.cpu().numpy())


def run_reference(args):
    rank, local_rank, world = dist_env()
    if rank != 0:
        return
    wl = WORKLOADS[args.workload]
    cb, t_sample = cpu_reference(wl, args.steps, args.warmup)
    line = {"impl": "reference", "metric": METRIC, "value": round(cb["value"], 4), "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": round(t_sample * 1e3, 1), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": {"workload": wl["name"], "l2": "n/a (CPU)"},
            "cpu_baseline": {**cb, "value": round(cb["value"], 4)},
            "e2e": {"value": round(cb["value"], 4), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def run_ours(args):
    rank, local_rank, world = dist_env()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the slam_b200 step has no CPU fallback (use --impl reference for the CPU baseline)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    from slam_llm_b200 import config as C, ops
    from slam_llm_b200.engine import SlamStepB200
    from slam_llm_b200.graphed import signature

    wl = WORKLOADS[args.workload]
    enc, llm = C.WHISPER[wl["enc"]], C.LLM[wl["llm"]]
    lora, proj = C.LoraCfg(wl["r"], wl["alpha"], tuple(wl["targets"])), C.ProjCfg("linear", 5, 2048)
    model, train_config = build_recipe_model(wl, enc, llm, lora, world)   # the recipe surface (setup_* + slam_model) builds the step
    eng = model.b200
    eng.defer_update = world > 1 and args.overlap == 1      # async gradient all-reduce, update applied behind the next step's frozen front end
    if wl["batch"] is None:
        if args.steps % wl["n_batches"]:
            raise SystemExit(f"--workload {args.workload}: --steps must be a multiple of {wl['n_batches']} (every step runs a different batch of the cycle)")
        dyn = make_dynamic_batches(wl, llm.vocab, seed=42 + rank, pin=True)
        host_batches = [b for b, _, _ in dyn]
        audio_s = sum(real for _, real, _ in dyn) / len(dyn)          # REAL audio seconds per step (mean over the cycle, this rank)
        padded_s = sum(pad for _, _, pad in dyn) / len(dyn)
        B, S = max(b["input_ids"].shape[0] for b in host_batches), max(b["input_ids"].shape[1] for b in host_batches)
    else:
        hb, S = make_batch(wl, llm.vocab, seed=42 + rank, pin=True)
        host_batches = [hb]
        B = wl["batch"]
        audio_s = padded_s = B * wl["seconds"]
    n_rows = 0
    for hb in host_batches:
        rows, tgts = SlamStepB200.label_rows(hb["labels"])
        hb["_rows"], hb["_targets"] = rows.pin_memory(), tgts.pin_memory()
        n_rows += rows.numel()
    n_rows //= len(host_batches)
    host_batch = host_batches[0]
    dev_batches = [{k: v.to(dev) for k, v in hb.items()} for hb in host_batches]
    dev_batch = dev_batches[0]
    counter = {"i": 0}
    lr = 1e-4

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    # one CUDA graph pair per shape bucket (slam_llm_b200/graphed.py); falls back to the eager step (and says so in `config`)
    graphs, launch_mode = {}, "eager (ctypes launches)"
    if args.graph == 1:
        try:
            from slam_llm_b200.graphed import GraphedTrainStep, signature
            for db in dev_batches:
                if signature(db) not in graphs:
                    graphs[signature(db)] = GraphedTrainStep(eng, db)
            launch_mode = f"cuda-graph replay (2 graphs/step, {len(graphs)} shape bucket(s)) + eager all-reduce/AdamW"
        except Exception as e:
            graphs = {}
            launch_mode = f"eager (graph capture failed: {type(e).__name__}: {e})"[:200]
            print("[bench] " + launch_mode, file=sys.stderr, flush=True)

    def run_step(b):
        g = graphs.get(signature(b)) if graphs else None
        if g is not None:
            return g.train_step(b, lr=lr, world_size=world)
        return eng.train_step(b, lr=lr, world_size=world)

    def step_resident():
        counter["i"] += 1
        return run_step(dev_batches[counter["i"] % len(dev_batches)])

    def step_e2e():
        counter["i"] += 1
        hb = host_batches[counter["i"] % len(host_batches)]
        g = graphs.get(signature(hb)) if graphs else None
        if g is not None:
            g.load(hb)                                                # pinned host -> the graph's static device buffers
            loss, acc = g.train_step(None, lr=lr, world_size=world)
        else:
            b = {k: v.to(dev, non_blocking=True) for k, v in hb.items()}
            loss, acc = eng.train_step(b, lr=lr, world_size=world)
        return loss.item()                                            # D2H read of the step's result

    if args.ncu_step:
        # profiling aid: `ncu --profile-from-start off ... python bench.py --ncu-step --graph 0` captures exactly ONE eager step
        for _ in range(3):
            eng.train_step(dev_batch, lr=lr, world_size=world)
        torch.cuda.synchronize()
        torch.cuda.profiler.start()
        eng.train_step(dev_batch, lr=lr, world_size=world)
        torch.cuda.synchronize()
        torch.cuda.profiler.stop()
        return
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    for _ in range(max(args.warmup, 3)):
        step_resident()
    # ---------------- timed region 1: inputs resident in HBM
    barrier()
    sampler.mark()
    l0 = ops.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        loss, acc = step_resident()
    eng.flush_update()                                                # deferred mode: the K-th update lands inside the timed region
    e1.record()
    barrier()
    launches = ops.launch_count() - l0                                # eager launches (all of the step, or only AdamW when graphed)
    if graphs:
        launches += args.steps * next(iter(graphs.values())).kernels_per_step   # + the kernels each graph replay launches
    ms = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms], device=dev)
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        ms = t.item()
    clocks = sampler.stop() if rank == 0 else None
    ms_per_step = ms / args.steps
    value = world * audio_s / (ms_per_step / 1e3)
    final_loss = loss.item()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, loss, acc, eng)              # before any later step overwrites the graph's loss buffer
    # ---------------- the same K steps again with a CUDA-event pair around every GEMM launch (roofline of the GEMM family);
    # kept out of the `value` region because ~900 extra event records per step cost ~3 % of host time
    for _ in range(2):                                               # the eager path's own allocator pool (the timed steps ran from graphs)
        eng.train_step(dev_batch, lr=lr, world_size=world)
    eng.flush_update()
    gemm_log = []
    ops.set_gemm_event_log(gemm_log)
    barrier()
    g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    g0.record()
    for _ in range(args.steps):
        counter["i"] += 1
        eng.train_step(dev_batches[counter["i"] % len(dev_batches)], lr=lr, world_size=world)   # eager: events cannot be read out of a graph replay
    eng.flush_update()
    g1.record()
    barrier()
    ops.set_gemm_event_log(None)
    ms_instr = g0.elapsed_time(g1)
    gemm_flops = sum(f for f, _, _ in gemm_log)
    gemm_ms = sum(a.elapsed_time(b) for _, a, b in gemm_log)

    # ---------------- timed region 2: end to end from pinned host buffers
    for _ in range(2):
        step_e2e()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        step_e2e()
    eng.flush_update()
    e1.record()
    barrier()
    ms2 = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms2], device=dev)
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        ms2 = t.item()
    e2e_value = world * audio_s / (ms2 / args.steps / 1e3)
    h2d = sum(v.numel() * v.element_size() for hb in host_batches for v in hb.values()) // len(host_batches)

    if args.breakdown:
        scale_breakdown(args, eng, dev_batch, lr, rank, world, dev)
    recipe = None
    if wl["batch"] is not None and not args.skip_recipe:          # every rank: the recipe loop under DDP is a collective affair
        try:
            recipe = recipe_leg(wl, model, train_config, llm, audio_s, args.steps, args.warmup, rank, local_rank, world)
        except Exception as e:
            recipe = {"unavailable": f"{type(e).__name__}: {e}"[:300]}
        eng.defer_update = world > 1 and args.overlap == 1
    if rank != 0:
        if world > 1:
            torch.distributed.destroy_process_group()
        return
    peak_tf, peak_hbm, peak_src = measured_peaks()
    fl = C.step_flops(enc, llm, proj, lora, B, int(padded_s / B * 100), S, n_label_rows=n_rows)
    achieved = gemm_flops / max(gemm_ms, 1e-9) / 1e9                  # TFLOP/s over all tcgen05 GEMM launches of the timed steps
    roof = {"bound": "tensor", "kernel": "gemm_tcgen05_kernel (all GEMM launches of the step: base, fused LoRA, dgrad, wgrad, lm_head)",
            "achieved": round(achieved, 1), "peak": peak_tf, "unit": "TFLOP/s", "frac": round(achieved / peak_tf, 4), "traffic": None,
            "peak_source": peak_src, "gemm_launches_per_step": len(gemm_log) // args.steps,
            "gemm_time_share_of_step": round(gemm_ms / ms_instr, 4),
            "measured_over": f"{args.steps} instrumented steps (CUDA events around every GEMM launch) run right after the timed region", "step_algorithmic_tflop": round(fl["total"] / 1e12, 2),
            "step_achieved_tflops": round(fl["total"] / (ms_per_step / 1e3) / 1e12, 1)}
    # DRAM bytes per GEMM launch: from the committed ncu pass over one eager step of this workload (tools/profile_round2.sh ->
    # tools/step_kernel_table.py); hardware counters cannot be read inside this process, so the number is per capture, not per run
    for traffic_file, key in (("r02c_step_kernels.json", ("gemm_family", "dram_bytes_per_launch")), ("r02b_step_kernels.json", ("gemm_family", "dram_bytes_per_launch")), ("r02_step_kernels.json", ("gemm_family", "dram_bytes_per_launch")),
                              ("r01_gemm_traffic.json", ("dram_bytes_per_launch",))):
        try:
            d = json.load(open(os.path.join(ROOT, "profiles", traffic_file)))
            for k in key:
                d = d[k]
            roof["traffic"], roof["traffic_source"] = d, "profiles/" + traffic_file
            break
        except Exception:
            continue
    eager = None
    if world == 1 and not args.skip_eager and wl["batch"] is not None:
        eager = eager_baseline(wl, enc, llm, lora, host_batch, dev, eng, audio_s, e2e_value, steps=args.steps, warmup=max(args.warmup, 3), model=model)
    cb = None
    if world == 1 and not args.skip_cpu:
        cb, _ = cpu_reference(wl, steps=2, warmup=0, budget_s=25.0)
        cb["value"] = round(cb["value"], 4)
    if world == 1 and not args.skip_traffic:
        torch.cuda.empty_cache()                                         # leave room for the child process's copy of the model
        try:
            traffic, how = measure_gemm_traffic(args.workload)
        except Exception as e:                                           # never let the diagnostic take the bench line down
            traffic, how = None, f"{type(e).__name__}: {e}"[:160]
        if traffic is not None:
            roof["traffic"], roof["traffic_source"] = traffic, how
        else:
            roof["traffic_source"] = f"{roof.get('traffic_source')} (in-run measurement unavailable: {how})"
    line = {"metric": METRIC, "value": round(value, 2), "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": round(ms_per_step, 3), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
            "data": "synthetic",
            "config": {"workload": wl["name"], "global_batch": B * world, "seq_len": S, "parallelism": f"dp{world}", "step_launch": launch_mode,
                       "audio_s_per_step_per_gpu": {"real": round(audio_s, 2), "padded": round(padded_s, 2)},
                       "grad_allreduce": ("none" if world == 1 else "async NCCL all-reduce of the flat fp32 arena, AdamW deferred behind the next step's frozen front end"
                                          if eng.defer_update else "blocking NCCL all-reduce of the flat fp32 arena"),
                       "l2": "per-step working set (35 GB bf16 weights streamed from HBM) >> 126 MB L2; no flush needed",
                       "lm_head_rows": "rows with a label only (loss/grad identical to full logits; eval path computes all rows)"},
            "clocks": clocks, "e2e": {"value": round(e2e_value, 2), "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
                                      "ms_per_step": round(ms2 / args.steps, 3)},
            "e2e_recipe": recipe, "gpu_launches": launches, "roofline": roof, "cpu_baseline": cb, "eager_gpu_baseline": eager, "loss": round(final_loss, 4)}
    print(json.dumps(line), flush=True)
    if world > 1:
        torch.distributed.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c3", choices=list(WORKLOADS))
    ap.add_argument("--skip-cpu", action="store_true", help="skip the cpu_baseline leg (profiling runs)")
    ap.add_argument("--skip-traffic", action="store_true", help="skip the in-run ncu child process that measures roofline.traffic (falls back to the committed ncu pass)")
    ap.add_argument("--ncu-step", action="store_true", help="run 3 warm-up steps, then ONE eager step between cudaProfilerStart/Stop, and exit")
    ap.add_argument("--graph", type=int, default=1, help="1 = replay the step from CUDA graphs (default), 0 = eager ctypes launches")
    ap.add_argument("--overlap", type=int, default=1, help="N>1: 1 = async all-reduce + deferred AdamW (default), 0 = blocking all-reduce")
    ap.add_argument("--breakdown", action="store_true", help="N>1 diagnostic: per-rank step time without / with blocking / with overlapped all-reduce "
                                                              "-> gpurun_out/scale_breakdown_n{N}.json")
    ap.add_argument("--skip-recipe", action="store_true", help="skip the e2e_recipe leg (train() + DataLoader)")
    ap.add_argument("--skip-eager", action="store_true", help="skip the eager-HF-on-GPU baseline leg (B-EAGER)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed to DIR/<name>.npy (loss, accuracy, sampled trainable parameters)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
