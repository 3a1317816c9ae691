"""Pin the oracle (and the host-side collator mirror) to outputs of the REFERENCE'S OWN code.

tests/golden/ref_*.pt were produced by tests/golden/make_ref_golden.py, which imports the original project's src/slam_llm unmodified
(datasets/speech_dataset.py __getitem__ + collator, models/slam_model.py setup_* + slam_model.forward, models/encoder.py,
models/projector.py, utils/metric.py, utils/config_utils.generate_peft_config) over HF LlamaForCausalLM and stand-ins for the
absent peft / openai-whisper packages (tests/ref_glue.py), runs one training step on the CPU and stores what came out.
These tests rebuild the same weights from the seeds, feed the oracle the same collated batch and require fp32-level agreement:
    loss rel <= 1e-5, activations / logits rel-max <= 1e-4, gradients rel-L2 <= 1e-4.
`make_ref_golden.py --check` re-runs the original code and compares it with the committed fixtures."""
import os
import sys

import pytest
import torch

import ref_fixture as rf
from oracle import slam_oracle as so

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FP32 = dict(loss=1e-5, act=1e-4, grad=1e-4)


def _oracle_vs_fixture(fix, small: bool):
    om = rf.oracle_model(fix)
    batch = rf.batch_of(fix)
    enc, llm, lora, proj = rf.cfgs(fix)
    mel = so.batch_log_mel(batch["audio_pcm"], enc.n_mels, batch.get("audio_pcm_lengths"))
    # log-mel: the reference run used the whisper stand-in with the filterbank from transformers.audio_utils (independent of the oracle's)
    assert tuple(mel.shape) == tuple(fix["mel"]["shape"])
    assert (mel.flatten()[: fix["mel"]["head"].numel()] - fix["mel"]["head"]).abs().max().item() < 5e-5
    assert abs(mel.norm().item() - fix["mel"]["norm"]) / fix["mel"]["norm"] < 1e-5
    c = fix["cfg"]
    ref = om.step(dict(batch), lr=c["lr"], weight_decay=c["wd"])
    assert abs(ref["loss"].item() - fix["loss"]) <= FP32["loss"] * abs(fix["loss"]), (ref["loss"].item(), fix["loss"])
    assert abs(float(ref["acc"]) - fix["acc"]) < 1e-7
    rows = rf.label_rows(batch["labels"])
    assert int(rows.sum()) == fix["n_labels"]
    lab = ref["logits"][:, :-1][rows]
    if small:
        assert rf.rel_max(ref["encoder_out"][:, :40], fix["encoder_out"]) < FP32["act"]
        assert rf.rel_max(ref["audio_tokens"][:, ::rf.AUDIO_TOKEN_STRIDE], fix["audio_tokens"]) < FP32["act"]
        assert rf.rel_max(lab, fix["label_logits"]) < FP32["act"]
        rf.check_probe(ref["inputs_embeds"], fix["inputs_embeds"], norm_rel=1e-5, head_rel=1e-4, what="inputs_embeds")
    else:
        rf.check_probe(ref["encoder_out"], fix["encoder_out"], norm_rel=1e-5, head_rel=1e-4, what="encoder_out")
        assert rf.rel_max(ref["encoder_out"][:, ::500, :64], fix["encoder_out_rows"]) < FP32["act"]
        rf.check_probe(ref["audio_tokens"], fix["audio_tokens"], norm_rel=1e-5, head_rel=1e-4, what="audio_tokens")
        rf.check_probe(lab, fix["label_logits"], norm_rel=1e-5, head_rel=1e-4, what="label_logits")
        assert rf.rel_max(lab[::20, :512], fix["label_logits_rows"]) < FP32["act"]
        clear = fix["label_margin"] > 1e-3
        assert torch.equal(lab.argmax(-1)[clear], fix["label_argmax"][clear])
    assert set(ref["grads"]) == set(fix["grads"])
    gmax = max((g["norm"] if rf.is_probe(g) else g.norm().item()) for g in fix["grads"].values())
    for k, g_ref in fix["grads"].items():
        g = ref["grads"][k]
        if rf.is_probe(g_ref):
            if g_ref["norm"] < 1e-6 * gmax:
                continue
            rf.check_probe(g, g_ref, norm_rel=FP32["grad"], head_rel=FP32["grad"] * 5, what=k)
        elif g_ref.norm().item() >= 1e-6 * gmax:
            assert rf.rel_l2(g, g_ref) < FP32["grad"], (k, rf.rel_l2(g, g_ref))
    # parameters after torch.optim.AdamW.step(): the first Adam step is ~ -lr*sign(g); only elements whose gradient is ~0 may differ
    after = om.trainable()
    for k, p in fix["after"].items():
        head = after[k].detach().flatten()[: p["head"].numel()]
        bad = ((head - p["head"]).abs() > 1e-6).float().mean().item()
        assert bad < 0.01, (k, bad)


@pytest.mark.parametrize("name", ["ref_tiny.pt", "ref_tiny_cov1d_all.pt", "ref_tiny_dynamic.pt"])
def test_oracle_matches_reference_run(name):
    _oracle_vs_fixture(rf.load(name), small=True)


@pytest.mark.skipif(os.environ.get("SLAM_SLOW_TESTS", "0") != "1", reason="2-3 min of CPU at Llama-3-8B widths: SLAM_SLOW_TESTS=1 (run when the fixture is regenerated)")
def test_oracle_matches_reference_run_at_real_widths():
    _oracle_vs_fixture(rf.load("ref_realwidth.pt"), small=False)


def test_oracle_s2s_matches_the_reference_s2s_model():
    """tests/golden/ref_s2s.pt = the reference's OWN examples/s2s/model/slam_model_s2s.py (forward + compute_parallel_loss) over HF Qwen2ForCausalLM,
    full fine-tune; the oracle's s2s_forward / s2s_step must reproduce loss, per-layer losses, accuracy and the gradient of every parameter."""
    fix = rf.load("ref_s2s.pt")
    c = fix["cfg"]
    L, TV, AV = c["code_layer"], c["text_vocab"], c["audio_vocab"]
    enc, llm, proj = so.EncoderCfg(*c["enc"]), so.LlmCfg(*c["llm"]), so.ProjCfg(*c["proj"])
    from parity_util import round_frozen
    om = round_frozen(so.OracleModel.build(enc, llm, None, proj, seed=c["seed"]))
    om.train_llm = True
    batch = so.s2s_synthetic_batch(2, 32000, L, TV, AV, seed=c["batch_seed"])
    ref = so.s2s_step(om, batch, L, TV, AV)
    assert abs(ref["loss"].item() - fix["loss"]) <= 1e-5 * abs(fix["loss"]), (ref["loss"].item(), fix["loss"])
    for got, want in zip(ref["layer_loss"], fix["layer_loss"]):
        assert abs(got.item() - want) <= 1e-5 * abs(want)
    assert abs(float(ref["acc"]) - fix["text_acc"]) < 1e-7
    rf.check_probe(ref["logits"], fix["logits"], norm_rel=1e-5, head_rel=1e-4, what="logits")
    assert set(ref["grads"]) == set(fix["grads"]), sorted(set(ref["grads"]) ^ set(fix["grads"]))
    gmax = max((g["norm"] if rf.is_probe(g) else g.norm().item()) for g in fix["grads"].values())
    for k, g_ref in fix["grads"].items():
        g = ref["grads"][k]
        if rf.is_probe(g_ref):
            if g_ref["norm"] >= 1e-6 * gmax:
                rf.check_probe(g, g_ref, norm_rel=1e-4, head_rel=5e-4, what=k)
        elif g_ref.norm().item() >= 1e-6 * gmax:
            assert rf.rel_l2(g, g_ref) < 1e-4, (k, rf.rel_l2(g, g_ref))


def test_realwidth_fixture_is_the_baseline_shape():
    fix = rf.load("ref_realwidth.pt")
    enc, llm, lora, proj = rf.cfgs(fix)
    full_e, full_l = so.WHISPER["large-v3"], so.LLM["llama-3-8b"]
    assert (enc.n_mels, enc.d, enc.heads) == (full_e.n_mels, full_e.d, full_e.heads) and enc.layers == 1
    assert (llm.vocab, llm.d, llm.heads, llm.kv_heads, llm.ffn, llm.rope_theta) == (full_l.vocab, full_l.d, full_l.heads, full_l.kv_heads, full_l.ffn, full_l.rope_theta)
    assert tuple(fix["batch"]["input_ids"].shape) == (2, 401) and fix["n_labels"] == 2 * 77


def test_collator_mirror_matches_reference_collator():
    """src/slam_llm/datasets/speech_dataset.py (this repo's host mirror) vs the reference collator's output on the same samples."""
    from slam_llm.datasets.speech_dataset import SpeechDatasetJsonl
    fix = rf.load("ref_collator.pt")
    ds = SpeechDatasetJsonl.__new__(SpeechDatasetJsonl)
    ds.tokenizer = type("T", (), {"pad_token_id": 2, "eos_token_id": 2})()
    ds.input_type, ds.inference_mode = "mel", False
    got = ds.collator([dict(s) for s in fix["samples"]])
    for k, v in fix["collated"].items():
        assert k in got and got[k] is not None, k
        if v.is_floating_point():
            assert torch.equal(got[k].float(), v.float()), k
        else:
            assert torch.equal(got[k].to(v.dtype), v), k
    for k in ("audio", "audio_mask"):
        assert got.get(k) is None


def test_dataset_mirror_reproduces_the_reference_batch(tmp_path):
    """WAV + jsonl -> this repo's SpeechDatasetJsonl (__getitem__ + collator) gives the ids / labels / masks the reference dataset gave
    (fixture `batch`), with raw PCM in place of the CPU mel (GPU front end) — and CPU mel items when b200_gpu_frontend=false."""
    import json
    import numpy as np
    from scipy.io import wavfile
    from slam_llm.datasets.speech_dataset import get_speech_dataset
    from omegaconf import OmegaConf
    sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
    from ref_glue import CharTokenizer
    fix = rf.load("ref_tiny.pt")
    utter = [(1.30, "hello world", "Transcribe. "), (2.05, "a b", "Transcribe speech to text. "), (0.70, "the quick brown fox", "Transcribe. ")]
    tok = CharTokenizer(512)
    for gpu_frontend in (True, False):
        samples, ds = [], None
        for i, ((_, target, prompt), p) in enumerate(zip(utter, fix["pcm_int16"])):
            wav = str(tmp_path / f"u{i}.wav")
            wavfile.write(wav, 16000, p.numpy().astype(np.int16))
            jl = str(tmp_path / f"u{i}.jsonl")
            with open(jl, "w") as f:
                f.write(json.dumps({"key": f"u{i}", "source": wav, "target": target}) + "\n")
            dc = OmegaConf.create(dict(train_data_path=jl, val_data_path=jl, prompt=prompt, mel_size=80, input_type="mel", b200_gpu_frontend=gpu_frontend))
            ds = get_speech_dataset(dc, tok, "train")
            samples.append(ds[0])
        got = ds.collator(samples)
        for k in ("input_ids", "labels", "attention_mask", "modality_mask"):
            assert torch.equal(got[k].to(fix["batch"][k].dtype), fix["batch"][k]), k
        assert torch.equal(got["audio_mel_post_mask"].float(), fix["batch"]["audio_mel_post_mask"].float())
        if gpu_frontend:
            assert got["audio_mel"] is None and torch.equal(got["audio_pcm"], rf.batch_of(fix)["audio_pcm"])
        else:
            assert got["audio_pcm"] is None
            assert (got["audio_mel"].flatten()[:512] - fix["mel"]["head"]).abs().max().item() < 5e-5


def test_dynamic_dataset_mirror_reproduces_the_reference_batches(tmp_path):
    """scp dir -> this repo's MultiTaskDataset / MultiTaskDynamicBatchDataset gives the same batches (window rule, ids, labels, masks) as the
    reference's, the too-long utterance dropped, PCM + lengths in place of the CPU mel with exactly the reference's padded mel width."""
    import json
    import numpy as np
    from scipy.io import wavfile
    from slam_llm.datasets.speech_dataset_large import get_speech_dataset
    from omegaconf import OmegaConf
    from ref_glue import CharTokenizer
    fix = rf.load("ref_tiny_dynamic.pt")
    dyn = fix["dynamic"]
    scp = tmp_path / "scp"
    scp.mkdir()
    with open(scp / "multitask.jsonl", "w") as f:
        for i, ((secs, task, target), p) in enumerate(zip(dyn["utts"], fix["all_pcm_int16"])):
            wav = str(tmp_path / f"d{i}.wav")
            wavfile.write(wav, 16000, p.numpy().astype(np.int16))
            f.write(json.dumps({"key": f"dyn{i}", "task": task, "target": target, "path": wav}) + "\n")
    pp = tmp_path / "prompts.jsonl"
    pp.write_text("".join(json.dumps({"task": t, "prompt": p}) + "\n" for t, p in dyn["prompts"].items()))
    dc = OmegaConf.create(dict(train_scp_file_path=str(scp), dev_scp_file_path=str(scp), test_scp_file_path=str(scp), multitask_prompt_path=str(pp),
                               append_info_tasks=[], prompt_style="USER: {}\n ASSISTANT:", mel_size=80, input_type="mel", pad_or_trim=False,
                               max_audio_length=dyn["max_audio_length"], train_max_frame_length=dyn["max_frame_length"],
                               eval_max_frame_length=dyn["max_frame_length"]))
    ds = get_speech_dataset(dc, CharTokenizer(512), "train")
    got = [ds.collator(items) for items in ds]
    assert len(got) == len(fix["all_batches"])
    for g, r in zip(got, fix["all_batches"]):
        for k in ("input_ids", "labels", "attention_mask", "modality_mask"):
            assert torch.equal(g[k].to(r[k].dtype), r[k]), k
        assert torch.equal(g["audio_mel_post_mask"].float(), r["audio_mel_post_mask"].float())
        assert g["audio_pcm"].shape[1] // 160 == 2 * r["audio_mel_post_mask"].shape[1] - (1 if (g["audio_pcm"].shape[1] // 160) % 2 else 0)
    picked = next(g for g, r in zip(got, fix["all_batches"]) if torch.equal(r["input_ids"], fix["batch"]["input_ids"]))
    want = rf.batch_of(fix)
    assert torch.equal(picked["audio_pcm"], want["audio_pcm"]) and torch.equal(picked["audio_pcm_lengths"], want["audio_pcm_lengths"])
    assert picked["audio_pcm"].shape[1] // 160 == fix["mel_frames"]


def test_audio_dataset_mirror_matches_the_reference_audio_dataset(tmp_path):
    """src/slam_llm/datasets/audio_dataset.py (EAT front end + item layout + collator; the aac_audiocaps recipes) vs what the reference's
    datasets/audio_dataset.py produced on the same WAV files (tests/golden/ref_audio_dataset.pt)."""
    import json
    import numpy as np
    from scipy.io import wavfile
    from slam_llm.datasets.audio_dataset import get_audio_dataset       # (importing slam_llm installs the omegaconf shim when needed)
    from omegaconf import OmegaConf
    from ref_glue import CharTokenizer
    fix = rf.load("ref_audio_dataset.pt")
    rows = []
    for i, (p, target) in enumerate(zip(fix["pcm_int16"], ("a dog barks", "rain", "birds are singing loudly"))):
        wav = str(tmp_path / f"a{i}.wav")
        wavfile.write(wav, 16000, p.numpy().astype(np.int16))
        rows.append({"key": f"aac{i}", "source": wav, "target": target})
    jl = tmp_path / "aac.jsonl"
    jl.write_text("\n".join(json.dumps(r) for r in rows))
    dc = OmegaConf.create(dict(train_data_path=str(jl), val_data_path=str(jl), prompt="Describe the audio you hear.", fix_length_audio=-1, input_type="mel",
                               model_name="eat", fbank_mean=-4.268, fbank_std=4.569, target_length=1024, fixed_length=False, random_crop=False,
                               encoder_projector_ds_rate=5, inference_mode=False))
    ds = get_audio_dataset(dc, CharTokenizer(1000), "train")
    items = [ds[i] for i in range(len(ds))]
    for got, want in zip(items, fix["items"]):
        assert got["audio_length"] == want["audio_length"] and got["target"] == want["target"]
        for k in ("input_ids", "labels", "attention_mask"):
            assert torch.equal(got[k], want[k]), k
        assert got["audio_mel"].shape == want["audio_mel"].shape and (got["audio_mel"] - want["audio_mel"]).abs().max().item() < 1e-5
    batch = ds.collator(items)
    for k, v in fix["collated"].items():
        if v.is_floating_point():
            assert (batch[k].float() - v.float()).abs().max().item() < 1e-5, k
        else:
            assert torch.equal(batch[k].to(v.dtype), v), k

