"""Run the REFERENCE'S OWN hot path on the CPU and commit what it produced (tests/golden/ref_*.pt).

    SLAM_LLM_REFERENCE=<checkout of the original SLAM-LLM> python tests/golden/make_ref_golden.py [--only NAME]   # writes ref_*.pt
    SLAM_LLM_REFERENCE=<checkout of the original SLAM-LLM> python tests/golden/make_ref_golden.py --check        # compares instead

Everything below `reference_step` executes the original project's src/slam_llm UNMODIFIED (imported through tests/ref_glue.py's
stand-ins for the absent third-party packages):
    datasets/speech_dataset.py  SpeechDatasetJsonl.__getitem__ + collator (:86-291)  on fabricated WAV + jsonl files
    models/slam_model.py        setup_encoder (:68-116) -> models/encoder.py WhisperWrappedEncoder.load (:9-45)
                                setup_llm (:118-221): AutoModelForCausalLM.from_pretrained + get_peft_model(generate_peft_config(...))
                                setup_encoder_projector (:223-236) -> models/projector.py
                                slam_model.forward (:283-407) incl. utils/metric.py compute_accuracy
    optimizer                   torch.optim.AdamW(model.parameters(), lr, weight_decay) as pipeline/finetune.py:247-251
The tests only read the committed fixtures (tests/test_ref_pinning.py, tests/test_ref_parity_gpu.py).  To keep every file small, a
tensor of more than FULL_MAX elements is stored as a probe (its norm and its first PROBE_HEAD elements), the parameters after the
AdamW step as probes of AFTER_HEAD elements, and the projector output of the small cases at every AUDIO_TOKEN_STRIDE-th token.

Weights come from the oracle's seeded initialisers (oracle/slam_oracle.py init_*) with the FROZEN matrices rounded to bf16
(what the device stores, tests/parity_util.round_frozen), so a test can rebuild identical weights from the seeds alone.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import tempfile

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, ROOT)

import ref_glue  # noqa: E402

ref_glue.install()                                   # the reference's src first on sys.path, stand-ins installed
from omegaconf import OmegaConf  # noqa: E402  (the repo shim or the real package)
from oracle import slam_oracle as so  # noqa: E402  (seeded initialisers + cfg dataclasses only; the arithmetic below is the reference's)
from parity_util import round_frozen  # noqa: E402
from ref_fixture import AUDIO_TOKEN_STRIDE  # noqa: E402

FULL_MAX, PROBE_HEAD, AFTER_HEAD = 4096, 2048, 1024

CASES = {
    # dh = 64, GQA 2:1, LoRA q/v, hidden 2048 (hard-coded in the reference projector, projector.py:11)
    "tiny": dict(enc=(80, 1500, 128, 2, 2), llm=(512, 256, 2, 4, 2, 512, 10000.0, 1e-5), lora=(8, 32, ("q_proj", "v_proj")),
                 proj=("linear", 5, 2048), seed=314, lr=1e-3, wd=0.01),
    # cov1d-linear projector + LoRA on all seven linears (aispeech_asr style), 128 mel bins, dh = 128
    "tiny_cov1d_all": dict(enc=(128, 1500, 128, 2, 1), llm=(640, 512, 2, 4, 1, 768, 500000.0, 1e-5), lora=(16, 32, so.LLM_LINEARS),
                           proj=("cov1d-linear", 5, 2048), seed=2718, lr=1e-3, wd=0.0),
    # BASELINE C3 widths at depth 1: Whisper-large-v3 widths x 1 layer + Llama-3-8B widths x 1 layer, B = 2, 30 s, S = 401
    "realwidth": dict(enc=(128, 1500, 1280, 20, 1), llm=(128256, 4096, 1, 32, 8, 14336, 500000.0, 1e-5), lora=(16, 32, ("q_proj", "v_proj")),
                      proj=("linear", 5, 2048), seed=1618, lr=1e-4, wd=0.0),
}
# dynamic-frame recipe (datasets/speech_dataset_large.py): natural-length utterances (odd and even frame counts), right padding only,
# batches formed by the window rule (:259-263) with a 260-token budget; the step runs on the first batch with >= 3 utterances
CASES["tiny_dynamic"] = dict(CASES["tiny"], seed=4242)
DYNAMIC = dict(max_frame_length=260, max_audio_length=3,
               utts=[(0.6131, "ASR", "ab"), (1.5075, "ST", "hello there"), (2.2506, "ASR", "c"), (0.9519, "ASR", "lorem ipsum"), (1.8107, "ST", "x y z"),
                     (3.1, "ASR", "dropped: longer than max_audio_length"), (0.4006, "ASR", "q")],
               prompts={"ASR": "Transcribe. ", "ST": "Translate the speech to German. "})

UTTERANCES = {   # (seconds, target text, prompt) — two prompts so the collator left-pads (speech_dataset.py:224-236)
    "tiny": [(1.30, "hello world", "Transcribe. "), (2.05, "a b", "Transcribe speech to text. "), (0.70, "the quick brown fox", "Transcribe. ")],
    "tiny_cov1d_all": [(0.9, "x", "Say it. "), (1.6, "lorem ipsum dolor", "Transcribe the speech. ")],
}


def cfgs(case):
    c = CASES[case]
    return so.EncoderCfg(*c["enc"]), so.LlmCfg(*c["llm"]), so.LoraCfg(c["lora"][0], c["lora"][1], tuple(c["lora"][2])), so.ProjCfg(*c["proj"])


def build_weights(case):
    enc, llm, lora, proj = cfgs(case)
    return round_frozen(so.OracleModel.build(enc, llm, lora, proj, seed=CASES[case]["seed"]))


def fabricate_pcm(case):
    g = torch.Generator().manual_seed(CASES[case]["seed"] + 7)
    out = []
    for secs, _, _ in UTTERANCES[case]:
        n = int(secs * 16000)
        out.append((torch.randn(n, generator=g) * 0.1 * 32768.0).round().clamp(-32768, 32767).to(torch.int16))
    return out


def reference_batch(case, tmp, mods, tokenizer):
    """WAV + jsonl on disk -> the reference dataset's __getitem__ and collator."""
    pcm = fabricate_pcm(case)
    n_mels = CASES[case]["enc"][0]
    samples, ds = [], None
    for i, ((secs, target, prompt), p) in enumerate(zip(UTTERANCES[case], pcm)):
        wav = os.path.join(tmp, f"utt{i}.wav")
        ref_glue.write_wav(wav, p.numpy())
        jl = os.path.join(tmp, f"utt{i}.jsonl")
        with open(jl, "w") as f:
            f.write(json.dumps({"key": f"utt{i}", "source": wav, "target": target}) + "\n")
        dc = OmegaConf.create(dict(train_data_path=jl, val_data_path=jl, prompt=prompt, mel_size=n_mels, input_type="mel"))
        ds = mods["speech_dataset"].get_speech_dataset(dc, tokenizer, "train")
        samples.append(ds[0])
    return ds.collator(samples), pcm


def dynamic_batches(case, tmp, mods, tokenizer):
    """scp dir + prompt file on disk -> the reference MultiTaskDataset / MultiTaskDynamicBatchDataset iteration and collator."""
    g = torch.Generator().manual_seed(CASES[case]["seed"] + 7)
    scp = os.path.join(tmp, "scp")
    os.makedirs(scp)
    pcm = []
    with open(os.path.join(scp, "multitask.jsonl"), "w") as f:
        for i, (secs, task, target) in enumerate(DYNAMIC["utts"]):
            n = int(round(secs * 16000))
            p = (torch.randn(n, generator=g) * 0.1 * 32768.0).round().clamp(-32768, 32767).to(torch.int16)
            pcm.append(p)
            wav = os.path.join(tmp, f"dyn{i}.wav")
            ref_glue.write_wav(wav, p.numpy())
            f.write(json.dumps({"key": f"dyn{i}", "task": task, "target": target, "path": wav}) + "\n")
    pp = os.path.join(tmp, "prompts.jsonl")
    with open(pp, "w") as f:
        for task, prompt in DYNAMIC["prompts"].items():
            f.write(json.dumps({"task": task, "prompt": prompt}) + "\n")
    dc = OmegaConf.create(dict(train_scp_file_path=scp, dev_scp_file_path=scp, test_scp_file_path=scp, multitask_prompt_path=pp, append_info_tasks=[],
                               prompt_style="USER: {}\n ASSISTANT:", mel_size=CASES[case]["enc"][0], input_type="mel", pad_or_trim=False,
                               max_audio_length=DYNAMIC["max_audio_length"],
                               train_max_frame_length=DYNAMIC["max_frame_length"], eval_max_frame_length=DYNAMIC["max_frame_length"]))
    ds = mods["speech_dataset_large"].get_speech_dataset(dc, tokenizer, "train")
    groups = [list(items) for items in ds]
    batches = [ds.collator(items) for items in groups]
    return batches, pcm


def synthetic_batch(case):
    """BASELINE-shaped batch (bench.make_batch layout) with the mel from the whisper stand-in."""
    import whisper
    _, llm, _, _ = cfgs(case)
    b = so.synthetic_batch(2, 480000, llm.vocab, prompt_len=24, answer_len=76, seed=CASES[case]["seed"] + 1)
    n_mels = CASES[case]["enc"][0]
    b["audio_mel"] = torch.stack([whisper.log_mel_spectrogram(w, n_mels=n_mels).permute(1, 0) for w in b["audio_pcm"]])
    return b


def build_reference_model(case, om, tmp, mods, tokenizer):
    from transformers import LlamaConfig, LlamaForCausalLM
    enc, llm, lora, proj = cfgs(case)
    # --- checkpoints on disk in the formats the reference loads
    wpt = os.path.join(tmp, "whisper_enc.pt")
    torch.save(ref_glue.whisper_checkpoint(om.enc_w, enc.n_mels, enc.n_ctx, enc.d, enc.heads, enc.layers), wpt)
    hf_dir = os.path.join(tmp, "llm")
    hc = LlamaConfig(vocab_size=llm.vocab, hidden_size=llm.d, intermediate_size=llm.ffn, num_hidden_layers=llm.layers, num_attention_heads=llm.heads,
                     num_key_value_heads=llm.kv_heads, rms_norm_eps=llm.eps, rope_theta=llm.rope_theta, max_position_embeddings=4096,
                     attention_bias=False, mlp_bias=False, tie_word_embeddings=False, hidden_act="silu", attn_implementation="eager")
    with torch.device("meta"):
        hf = LlamaForCausalLM(hc)
    hf = hf.to_empty(device="cpu")
    missing, unexpected = hf.load_state_dict(om.llm_w, strict=False)
    assert not unexpected and all("rotary" in m or "inv_freq" in m for m in missing), (missing, unexpected)
    if hasattr(hf.model, "rotary_emb"):                                               # buffers are not in the state dict: rebuild
        hf.model.rotary_emb = type(hf.model.rotary_emb)(config=hc)
    hf.save_pretrained(hf_dir, safe_serialization=True)
    del hf
    train_config = OmegaConf.create(dict(enable_fsdp=False, enable_ddp=False, low_cpu_fsdp=False, quantization=False, use_fast_kernels=False,
                                         freeze_llm=True, freeze_encoder=True, use_peft=True,
                                         peft_config=dict(peft_method="lora", r=lora.r, lora_alpha=lora.alpha, target_modules=list(lora.targets),
                                                          bias="none", task_type="CAUSAL_LM", lora_dropout=0.0, inference_mode=False)))
    model_config = OmegaConf.create(dict(llm_name="llama", llm_path=hf_dir, llm_dim=llm.d, encoder_name="whisper", encoder_path=wpt, encoder_path_hf=None,
                                         whisper_decode=False, encoder_dim=enc.d, encoder_projector=proj.kind, encoder_projector_ds_rate=proj.k))
    sm = mods["slam_model"]

    class _AutoCausalLM435:
        """transformers 4.35.2 (the reference's pin) accepted `load_in_8bit=None, device_map=None, use_cache=None` and defaulted to eager
        attention; 5.5.0 validates config fields strictly.  Same call, None-valued kwargs dropped, eager attention requested."""
        @staticmethod
        def from_pretrained(path, **kw):
            from transformers import AutoModelForCausalLM
            return AutoModelForCausalLM.from_pretrained(path, attn_implementation="eager", torch_dtype=torch.float32,
                                                        **{k: v for k, v in kw.items() if v is not None})
    sm.AutoModelForCausalLM = _AutoCausalLM435
    encoder = sm.setup_encoder(train_config, model_config)
    llm_mod = sm.setup_llm(train_config, model_config)
    projector = sm.setup_encoder_projector(train_config, model_config)
    model = sm.slam_model(encoder, llm_mod, projector, tokenizer, train_config, model_config)
    # seeded trainables (peft would zero-init B: dA would vanish, SURVEY §7)
    sd = {f"llm.base_model.model.{k}": v for k, v in om.lora_w.items()}
    sd.update({f"encoder_projector.{k}": v for k, v in om.proj_w.items()})
    missing, unexpected = model.load_state_dict(sd, strict=False)
    assert not unexpected, unexpected
    trainable = {n for n, p in model.named_parameters() if p.requires_grad}
    assert trainable == set(sd), (sorted(trainable ^ set(sd))[:6])
    return model


S2S = dict(code_layer=3, text_vocab=400, audio_vocab=80, enc=(80, 1500, 128, 2, 1), llm=(640, 256, 2, 4, 1, 384, 1000000.0, 1e-6, True, True),
           proj=("linear", 5, 2048), seed=21, batch_seed=5)


def reference_s2s_step() -> dict:
    """The reference's OWN SLAM-Omni model class (examples/s2s/model/slam_model_s2s.py: forward :160-283 + compute_parallel_loss :285-306) over
    an HF Qwen2ForCausalLM built by the reference's setup_llm with freeze_llm=false (full fine-tune), the reference encoder / projector
    factories, on the oracle's synthetic s2s batch (CPU mel from the whisper stand-in)."""
    import importlib
    import whisper
    from transformers import Qwen2Config, Qwen2ForCausalLM
    mods = ref_glue.reference_modules()
    sys.path.insert(0, os.path.join(ref_glue.REFERENCE, "examples", "s2s"))
    s2s_mod = importlib.import_module("model.slam_model_s2s")
    assert s2s_mod.__file__.startswith(os.path.abspath(ref_glue.REFERENCE))
    L, TV, AV = S2S["code_layer"], S2S["text_vocab"], S2S["audio_vocab"]
    enc, llm, proj = so.EncoderCfg(*S2S["enc"]), so.LlmCfg(*S2S["llm"]), so.ProjCfg(*S2S["proj"])
    assert llm.vocab == TV + L * AV
    om = round_frozen(so.OracleModel.build(enc, llm, None, proj, seed=S2S["seed"]))
    torch.manual_seed(0)
    with tempfile.TemporaryDirectory() as tmp:
        wpt = os.path.join(tmp, "whisper_enc.pt")
        torch.save(ref_glue.whisper_checkpoint(om.enc_w, enc.n_mels, enc.n_ctx, enc.d, enc.heads, enc.layers), wpt)
        hf_dir = os.path.join(tmp, "llm")
        hc = Qwen2Config(vocab_size=llm.vocab, hidden_size=llm.d, intermediate_size=llm.ffn, num_hidden_layers=llm.layers, num_attention_heads=llm.heads,
                         num_key_value_heads=llm.kv_heads, rms_norm_eps=llm.eps, rope_theta=llm.rope_theta, tie_word_embeddings=True,
                         max_position_embeddings=4096, use_sliding_window=False, attn_implementation="eager")
        hf = Qwen2ForCausalLM(hc)
        missing, unexpected = hf.load_state_dict(om.llm_w, strict=False)
        assert not unexpected and set(missing) <= {"lm_head.weight"}, (missing, unexpected)
        hf.save_pretrained(hf_dir, safe_serialization=True)
        del hf
        train_config = OmegaConf.create(dict(enable_fsdp=False, enable_ddp=False, low_cpu_fsdp=False, quantization=False, use_fast_kernels=False,
                                             freeze_llm=False, freeze_encoder=True, use_peft=False, task_type="s2s"))
        model_config = OmegaConf.create(dict(llm_name="qwen2", llm_path=hf_dir, llm_dim=llm.d, encoder_name="whisper", encoder_path=wpt,
                                             encoder_path_hf=None, whisper_decode=False, encoder_dim=enc.d, encoder_projector=proj.kind,
                                             encoder_projector_ds_rate=proj.k,
                                             vocab_config=dict(code_layer=L, padded_text_vocabsize=TV, padded_audio_vocabsize=AV, total_vocabsize=llm.vocab)))
        sm = mods["slam_model"]

        class _AutoCausalLM435:
            @staticmethod
            def from_pretrained(path, **kw):
                from transformers import AutoModelForCausalLM
                return AutoModelForCausalLM.from_pretrained(path, attn_implementation="eager", torch_dtype=torch.float32,
                                                            **{k: v for k, v in kw.items() if v is not None})
        sm.AutoModelForCausalLM = _AutoCausalLM435
        encoder = sm.setup_encoder(train_config, model_config)
        llm_mod = sm.setup_llm(train_config, model_config)
        projector = sm.setup_encoder_projector(train_config, model_config)
        model = s2s_mod.slam_model_s2s(encoder, llm_mod, projector, None, None, None, None, None, train_config, model_config)
    sd = {f"encoder_projector.{k}": v for k, v in om.proj_w.items()}
    missing, unexpected = model.load_state_dict(sd, strict=False)
    assert not unexpected
    model.train()
    batch = so.s2s_synthetic_batch(2, 32000, L, TV, AV, seed=S2S["batch_seed"])
    mel = torch.stack([whisper.log_mel_spectrogram(w, n_mels=enc.n_mels).permute(1, 0) for w in batch["audio_pcm"]])
    feed = dict(input_ids=batch["input_ids"].clone(), attention_mask=batch["attention_mask"], labels=batch["labels"], modality_mask=batch["modality_mask"],
                audio_mel=mel)
    outputs, text_acc, audio_acc, layer_loss = model(**feed)
    outputs.loss.backward()
    trainable = {n: p for n, p in model.named_parameters() if p.requires_grad}
    grads = {}
    for n, p in trainable.items():
        if n == "llm.lm_head.weight":                                   # tied: the same tensor as the embedding (HF lists it once)
            continue
        g = p.grad.detach() if p.grad is not None else torch.zeros_like(p)
        grads[n] = g.clone() if g.numel() <= FULL_MAX else probe(g, PROBE_HEAD)
    return dict(case="s2s", cfg=S2S, loss=outputs.loss.item(), text_acc=float(text_acc), layer_loss=[float(l) for l in layer_loss], grads=grads,
                mel=probe(mel, 512), logits=probe(outputs.logits.detach(), 2048), trainable=sorted(grads))


def probe(t: torch.Tensor, n: int = 256):
    t = t.detach().float()
    return dict(norm=t.norm().item(), head=t.flatten()[:n].clone(), shape=tuple(t.shape))


def reference_step(case: str) -> dict:
    mods = ref_glue.reference_modules()
    enc, llm, lora, proj = cfgs(case)
    om = build_weights(case)
    tokenizer = ref_glue.CharTokenizer(llm.vocab)
    torch.manual_seed(0)
    with tempfile.TemporaryDirectory() as tmp:
        all_batches = None
        if case == "tiny_dynamic":
            all_batches, pcm_all = dynamic_batches(case, tmp, mods, tokenizer)
            pick = next(i for i, b in enumerate(all_batches) if b["input_ids"].shape[0] >= 3)
            batch = all_batches[pick]
            used, seen = [], 0                                       # utterances of the picked batch, in dataset order (the too-long one is dropped)
            kept = [i for i, (secs, _, _) in enumerate(DYNAMIC["utts"]) if secs <= DYNAMIC["max_audio_length"]]
            for bi, b in enumerate(all_batches):
                n = b["input_ids"].shape[0]
                if bi == pick:
                    used = kept[seen: seen + n]
                seen += n
            pcm = [pcm_all[i] for i in used]
        elif case in UTTERANCES:
            batch, pcm = reference_batch(case, tmp, mods, tokenizer)
        else:
            batch, pcm = synthetic_batch(case), None
        model = build_reference_model(case, om, tmp, mods, tokenizer)
    model.train()                                                                      # utils/train_utils.py:92
    feed = {k: (v.clone() if torch.is_tensor(v) else v) for k, v in batch.items() if k != "audio_pcm"}
    with torch.no_grad():
        enc_out = model.encoder.extract_variable_length_features(feed["audio_mel"].permute(0, 2, 1))
        aud = model.encoder_projector(enc_out)
        embeds, _ = model(**{k: (v.clone() if torch.is_tensor(v) else v) for k, v in feed.items()}, inference_mode=True)
    outputs, acc = model(**feed)                                                       # forward() edits input_ids in place: `feed` holds clones
    outputs.loss.backward()
    grads = {n: p.grad.detach().clone() for n, p in model.named_parameters() if p.requires_grad}
    c = CASES[case]
    optimizer = torch.optim.AdamW(model.parameters(), lr=c["lr"], weight_decay=c["wd"])   # pipeline/finetune.py:247-251
    optimizer.step()
    after = {n: p.detach().clone() for n, p in model.named_parameters() if p.requires_grad}
    labels = batch["labels"]
    rows = (labels[:, 1:] != -100)
    lab_logits = outputs.logits.detach()[:, :-1][rows]                                 # logits of the rows that carry a label
    out = dict(case=case, cfg=dict(enc=c["enc"], llm=c["llm"], lora=c["lora"], proj=c["proj"], seed=c["seed"], lr=c["lr"], wd=c["wd"]),
               loss=outputs.loss.item(), acc=float(acc), n_labels=int(rows.sum()),
               batch={k: v.clone() for k, v in batch.items() if torch.is_tensor(v) and k not in ("audio_mel", "audio_pcm")})
    if all_batches is not None:
        out["all_batches"] = [{k: v.clone() for k, v in b.items() if torch.is_tensor(v) and k != "audio_mel"} for b in all_batches]
        out["all_pcm_int16"] = pcm_all
        out["dynamic"] = DYNAMIC
        out["mel_frames"] = int(batch["audio_mel"].shape[1])
    if pcm is not None:
        out["pcm_int16"] = pcm
    else:
        out["batch_seed"] = c["seed"] + 1
    small = case != "realwidth"
    out["mel"] = probe(batch["audio_mel"], 512)
    if small:
        out["encoder_out"] = enc_out[:, :40].clone()                                   # first 40 frames of every utterance, all channels
        out["audio_tokens"] = aud[:, ::AUDIO_TOKEN_STRIDE].clone()
        out["inputs_embeds"] = probe(embeds, 1024)
        out["label_logits"] = lab_logits.clone()
        out["grads"] = {k: (v.clone() if v.numel() <= FULL_MAX else probe(v, PROBE_HEAD)) for k, v in grads.items()}
        out["after"] = {k: probe(v, AFTER_HEAD) for k, v in after.items()}
    else:
        out["encoder_out"] = probe(enc_out)
        out["encoder_out_rows"] = enc_out[:, ::500, :64].clone()
        out["audio_tokens"] = probe(aud)
        out["inputs_embeds"] = probe(embeds)
        out["label_logits"] = probe(lab_logits)
        out["label_logits_rows"] = lab_logits[::20, :512].clone()
        out["label_argmax"] = lab_logits.argmax(-1).clone()
        top2 = lab_logits.topk(2, dim=-1).values
        out["label_margin"] = (top2[:, 0] - top2[:, 1]).clone()                        # argmax is only comparable where the margin is clear
        out["grads"] = {k: probe(v) for k, v in grads.items()}
        out["after"] = {k: probe(v) for k, v in after.items()}
    return out


def collator_cases() -> dict:
    """The reference collators alone, on token-level inputs (no audio decode): jsonl collator with mixed prompt/answer lengths."""
    mods = ref_glue.reference_modules()
    tok = ref_glue.CharTokenizer(1000)
    ds = mods["speech_dataset"].SpeechDatasetJsonl.__new__(mods["speech_dataset"].SpeechDatasetJsonl)
    ds.tokenizer, ds.IGNORE_INDEX, ds.input_type, ds.inference_mode = tok, -100, "mel", False
    g = torch.Generator().manual_seed(5)
    samples = []
    for audio_length, prompt_length, answer_length, frames in ((7, 5, 4, 70), (3, 9, 1, 31), (12, 2, 8, 120), (1, 1, 1, 9)):
        n = audio_length + prompt_length + answer_length
        ids = torch.randint(3, 1000, (n,), generator=g)
        ids[:audio_length] = -1
        labels = ids.clone()
        labels[:audio_length + prompt_length] = -100
        samples.append(dict(input_ids=ids, labels=labels, attention_mask=ids.ge(-1), audio=None, audio_mel=torch.randn(frames, 8, generator=g),
                            audio_length=audio_length, prompt_length=prompt_length))
    out = ds.collator(samples)
    return dict(samples=samples, collated={k: v for k, v in out.items() if v is not None})


def audio_dataset_case() -> dict:
    """The reference's datasets/audio_dataset.py (EAT front end: models/EAT/EAT.py EAT_preprocess + item layout + collator) on fabricated WAVs."""
    import importlib
    ref_glue.install()
    mod = importlib.import_module("slam_llm.datasets.audio_dataset")
    assert mod.__file__.startswith(ref_glue.REFERENCE_SRC)

    def _wav_load(path, *a, **kw):
        """torchaudio.load needs torchcodec in torchaudio 2.11 (absent offline): 16-bit PCM WAV through scipy, same return convention
        ([channels, n] float32 in [-1, 1), sample rate)."""
        from scipy.io import wavfile
        rate, data = wavfile.read(path)
        return torch.from_numpy(data.astype("float32") / 32768.0).reshape(1, -1), rate
    mod.torchaudio.load = _wav_load
    tok = ref_glue.CharTokenizer(1000)
    g = torch.Generator().manual_seed(77)
    pcm, samples = [], []
    with tempfile.TemporaryDirectory() as tmp:
        rows = []
        for i, (secs, target) in enumerate(((1.234, "a dog barks"), (2.5, "rain"), (0.8, "birds are singing loudly"))):
            p = (torch.randn(int(secs * 16000), generator=g) * 0.1 * 32768.0).round().clamp(-32768, 32767).to(torch.int16)
            pcm.append(p)
            wav = os.path.join(tmp, f"aac{i}.wav")
            ref_glue.write_wav(wav, p.numpy())
            rows.append({"key": f"aac{i}", "source": wav, "target": target})
        jl = os.path.join(tmp, "aac.jsonl")
        with open(jl, "w") as f:
            f.write("\n".join(json.dumps(r) for r in rows))
        dc = OmegaConf.create(dict(train_data_path=jl, val_data_path=jl, prompt="Describe the audio you hear.", fix_length_audio=-1, input_type="mel",
                                   model_name="eat", fbank_mean=-4.268, fbank_std=4.569, target_length=1024, fixed_length=False, random_crop=False,
                                   encoder_projector_ds_rate=5, inference_mode=False))
        ds = mod.get_audio_dataset(dc, tok, "train")
        samples = [ds[i] for i in range(len(ds))]
        batch = ds.collator(samples)
    return dict(pcm_int16=pcm, items=[{k: v for k, v in s.items() if torch.is_tensor(v) or isinstance(v, (int, str))} for s in samples],
                collated={k: v for k, v in batch.items() if torch.is_tensor(v)})


def _cmp(a, b, path=""):
    if isinstance(a, dict):
        assert set(a) == set(b), (path, set(a) ^ set(b))
        for k in a:
            _cmp(a[k], b[k], f"{path}/{k}")
    elif isinstance(a, (list, tuple)):
        assert len(a) == len(b), path
        for i, (x, y) in enumerate(zip(a, b)):
            _cmp(x, y, f"{path}[{i}]")
    elif torch.is_tensor(a):
        if a.is_floating_point():
            assert torch.allclose(a, b, rtol=1e-4, atol=1e-6), (path, (a - b).abs().max().item())
        else:
            assert torch.equal(a, b), path
    elif isinstance(a, float):
        assert abs(a - b) <= 1e-5 * max(1.0, abs(a)), (path, a, b)
    else:
        assert a == b, (path, a, b)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--check", action="store_true")
    ap.add_argument("--only", default=None)
    args = ap.parse_args()
    todo = {f"ref_{c}.pt": (lambda c=c: reference_step(c)) for c in CASES}
    todo["ref_collator.pt"] = collator_cases
    todo["ref_s2s.pt"] = reference_s2s_step
    todo["ref_audio_dataset.pt"] = audio_dataset_case
    for name, fn in todo.items():
        if args.only and args.only not in name:
            continue
        out = fn()
        path = os.path.join(HERE, name)
        if args.check:
            _cmp(torch.load(path), out, name)
            print("ok", name)
        else:
            torch.save(out, path)
            print("wrote", name, os.path.getsize(path), "bytes", {k: out[k] for k in ("loss", "acc", "n_labels") if k in out})


if __name__ == "__main__":
    main()
