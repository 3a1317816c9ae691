"""Helpers shared by the CPU pinning tests and the GPU parity tests that read the REFERENCE-RUN fixtures
(tests/golden/ref_*.pt, produced by tests/golden/make_ref_golden.py from the original project's own code).  Test infrastructure."""
from __future__ import annotations

import os

import torch

from oracle import slam_oracle as so
from parity_util import round_frozen

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
AUDIO_TOKEN_STRIDE = 10          # the small fixtures keep every 10th projector output token (audio_tokens[:, ::10]) to stay small


def load(name: str) -> dict:
    return torch.load(os.path.join(GOLDEN, name), weights_only=False)


def cfgs(fix):
    c = fix["cfg"]
    return (so.EncoderCfg(*c["enc"]), so.LlmCfg(*c["llm"]), so.LoraCfg(c["lora"][0], c["lora"][1], tuple(c["lora"][2])), so.ProjCfg(*c["proj"]))


def oracle_model(fix):
    """Identical weights to the ones the reference run used: the oracle's seeded initialisers, frozen matrices rounded to bf16."""
    enc, llm, lora, proj = cfgs(fix)
    return round_frozen(so.OracleModel.build(enc, llm, lora, proj, seed=fix["cfg"]["seed"]))


def batch_of(fix) -> dict:
    """The batch the reference collator produced (ids / labels / masks from the fixture) + the raw waveforms (`audio_pcm`, 30 s padded,
    what whisper.load_audio + pad_or_trim fed the reference's log-mel)."""
    b = {k: v.clone() for k, v in fix["batch"].items() if k in ("input_ids", "labels", "attention_mask", "modality_mask")}
    if "pcm_int16" in fix:
        dynamic = "dynamic" in fix                                   # natural lengths, right-padded to the longest (speech_dataset_large.py)
        width = max(p.numel() for p in fix["pcm_int16"]) if dynamic else 480000
        pcm = torch.zeros(len(fix["pcm_int16"]), width)
        for i, p in enumerate(fix["pcm_int16"]):
            pcm[i, : p.numel()] = p.float() / 32768.0
        b["audio_pcm"] = pcm
        if dynamic:
            b["audio_pcm_lengths"] = torch.tensor([p.numel() for p in fix["pcm_int16"]], dtype=torch.int32)
    else:
        _, llm, _, _ = cfgs(fix)
        syn = so.synthetic_batch(b["input_ids"].shape[0], 480000, llm.vocab, prompt_len=24, answer_len=76, seed=fix["batch_seed"])
        for k in ("input_ids", "labels", "attention_mask", "modality_mask"):
            assert torch.equal(syn[k], b[k]), k                      # the seeded generator reproduces the committed batch
        b["audio_pcm"] = syn["audio_pcm"]
    b["input_ids"] = b["input_ids"].clone()
    return b


def label_rows(labels: torch.Tensor) -> torch.Tensor:
    return labels[:, 1:] != -100


def rel_l2(a, b) -> float:
    a, b = a.detach().float().cpu(), b.detach().float().cpu()
    return ((a - b).norm() / b.norm().clamp_min(1e-30)).item()


def rel_max(a, b) -> float:
    a, b = a.detach().float().cpu(), b.detach().float().cpu()
    return ((a - b).abs().max() / b.abs().max().clamp_min(1e-30)).item()


def cosine(a, b) -> float:
    a, b = a.detach().float().cpu().flatten(), b.detach().float().cpu().flatten()
    return torch.nn.functional.cosine_similarity(a, b, dim=0).item()


def is_probe(x) -> bool:
    return isinstance(x, dict) and "norm" in x and "head" in x


def check_probe(t: torch.Tensor, p: dict, *, norm_rel: float, head_cos: float = None, head_rel: float = None, what: str = ""):
    t = t.detach().float().cpu()
    assert tuple(t.shape) == tuple(p["shape"]), (what, t.shape, p["shape"])
    assert abs(t.norm().item() - p["norm"]) <= norm_rel * max(p["norm"], 1e-12), (what, "norm", t.norm().item(), p["norm"])
    head = t.flatten()[: p["head"].numel()]
    if head_cos is not None and p["head"].norm().item() > 1e-6 * max(p["norm"], 1e-30):
        assert cosine(head, p["head"]) >= head_cos, (what, "head cosine", cosine(head, p["head"]))
    if head_rel is not None:
        assert rel_l2(head, p["head"]) <= head_rel, (what, "head rel-l2", rel_l2(head, p["head"]))
