"""CUDA step (through the C ABI) vs outputs of the REFERENCE'S OWN code run on the CPU (tests/golden/ref_*.pt; generator
tests/golden/make_ref_golden.py, pinned oracle == fixture in tests/test_ref_pinning.py).

Tolerances (bf16 compute / fp32 accumulate vs the reference's fp32; BASELINE.md §4, written here):
    log-mel abs <= 2e-3 on the (x+4)/4 scale;  activations / logits rel-max <= 2e-2 and cosine >= 0.999;  loss rel <= 5e-3;
    gradients cosine >= 0.99 and rel-L2 <= 3e-2 (per tensor with non-negligible norm);  accuracy equal wherever the reference's
    top-1 margin is clear of bf16 noise.
The real-width case (Whisper-large-v3 widths x 1 layer + Llama-3-8B widths x 1 layer, B = 2, S = 401) exercises every GEMM / attention /
CE shape of the BASELINE config (D 4096, F 14336, V 128256, 32/8 heads dh 128, d 1280 / 20 heads, T' 1500) against the reference."""
import pytest
import torch

import ref_fixture as rf

pytestmark = pytest.mark.gpu


def build_engine(fix, om):
    from slam_llm_b200 import config as C
    from slam_llm_b200.engine import SlamStepB200
    enc, llm, lora, proj = rf.cfgs(fix)
    return SlamStepB200(C.EncoderCfg(**vars(enc)), C.LlmCfg(**vars(llm)), C.LoraCfg(lora.r, lora.alpha, tuple(lora.targets), lora.dropout),
                        C.ProjCfg(**vars(proj)), device="cuda:0", enc_weights=om.enc_w, llm_weights=om.llm_w, lora_weights=om.lora_w,
                        proj_weights=om.proj_w)


def _step_vs_fixture(fix, small: bool):
    om = rf.oracle_model(fix)                      # weights only (seeded initialisers); the expected values are the reference run's
    eng = build_engine(fix, om)
    batch = rf.batch_of(fix)
    gb = {k: v.cuda() for k, v in batch.items()}
    mel = eng.log_mel(gb["audio_pcm"], gb.get("audio_pcm_lengths"))
    assert tuple(mel.shape) == tuple(fix["mel"]["shape"])
    assert (mel.flatten()[: fix["mel"]["head"].numel()].cpu() - fix["mel"]["head"]).abs().max().item() < 2e-3
    assert abs(mel.norm().item() - fix["mel"]["norm"]) / fix["mel"]["norm"] < 2e-3
    enc_out = eng.encoder.forward(mel)
    aud = eng.projector.forward(enc_out, save=False)
    if small:
        assert rf.rel_max(enc_out[:, :40], fix["encoder_out"]) < 2e-2 and rf.cosine(enc_out[:, :40], fix["encoder_out"]) > 0.999
        aud = aud[:, ::rf.AUDIO_TOKEN_STRIDE]
        assert rf.rel_max(aud, fix["audio_tokens"]) < 2e-2 and rf.cosine(aud, fix["audio_tokens"]) > 0.999
    else:
        rf.check_probe(enc_out, fix["encoder_out"], norm_rel=1e-2, head_cos=0.999, what="encoder_out")
        rows = enc_out[:, ::500, :64]
        assert rf.rel_max(rows, fix["encoder_out_rows"]) < 2e-2 and rf.cosine(rows, fix["encoder_out_rows"]) > 0.999
        rf.check_probe(aud, fix["audio_tokens"], norm_rel=1e-2, head_cos=0.999, what="audio_tokens")

    loss, acc, _ = eng.forward(gb, train=True)
    assert abs(loss.item() - fix["loss"]) <= 5e-3 * abs(fix["loss"]), (loss.item(), fix["loss"])
    lab = eng._ctx["logits"].float().cpu()          # fp32 logits of the rows that carry a label, in (b, s) order like logits[:, :-1][rows]
    assert lab.shape[0] == fix["n_labels"]
    if small:
        assert rf.rel_max(lab, fix["label_logits"]) < 2e-2 and rf.cosine(lab, fix["label_logits"]) > 0.999
        top2 = fix["label_logits"].topk(2, dim=-1).values
        margin, ref_arg = top2[:, 0] - top2[:, 1], fix["label_logits"].argmax(-1)
    else:
        rf.check_probe(lab, fix["label_logits"], norm_rel=1e-2, head_cos=0.999, what="label_logits")
        sub = lab[::20, :512]
        assert rf.rel_max(sub, fix["label_logits_rows"]) < 2e-2 and rf.cosine(sub, fix["label_logits_rows"]) > 0.999
        margin, ref_arg = fix["label_margin"], fix["label_argmax"]
    clear = margin > 4e-2 * lab.abs().max().item()                                    # twice the activation tolerance
    assert torch.equal(lab.argmax(-1)[clear], ref_arg[clear])
    if bool(clear.all()):
        assert abs(acc.item() - fix["acc"]) < 1e-6

    eng.backward()
    grads = eng.trainable_state("grad")
    assert set(grads) == set(fix["grads"])
    gmax = max((g["norm"] if rf.is_probe(g) else g.norm().item()) for g in fix["grads"].values())
    checked = 0
    for k, g_ref in fix["grads"].items():
        g = grads[k]
        if rf.is_probe(g_ref):
            if g_ref["norm"] < 1e-3 * gmax:
                continue
            rf.check_probe(g, g_ref, norm_rel=3e-2, head_cos=0.99, what=k)
        else:
            if g_ref.norm().item() < 1e-3 * gmax:
                continue
            assert rf.cosine(g, g_ref) > 0.99, (k, rf.cosine(g, g_ref))
            assert rf.rel_l2(g, g_ref) < (4e-2 if "conv1d" in k else 3e-2), (k, rf.rel_l2(g, g_ref))
        checked += 1
    assert checked >= (4 if not small else 6), checked

    # AdamW (pipeline/finetune.py:247-251) through slam_adamw: first step ~ -lr*sign(g); elements whose gradient is bf16-noise may flip
    c = fix["cfg"]
    before = {k: v.clone() for k, v in eng.trainable_state().items()}
    eng.optimizer_step(c["lr"], c["wd"])
    after = eng.trainable_state()
    for k, p in fix["after"].items():
        n = p["head"].numel()
        g_ref = fix["grads"][k]
        upd = (after[k].flatten()[:n] - before[k].flatten()[:n]).cpu()
        upd_ref = p["head"] - before[k].flatten()[:n].cpu()
        if upd_ref.norm().item() > 0 and (g_ref["norm"] if rf.is_probe(g_ref) else g_ref.norm().item()) >= 1e-3 * gmax:
            assert rf.cosine(upd, upd_ref) > 0.9, (k, rf.cosine(upd, upd_ref))


@pytest.mark.parametrize("name", ["ref_tiny.pt", "ref_tiny_cov1d_all.pt", "ref_tiny_dynamic.pt"])
def test_cuda_step_matches_reference_run(name):
    """ref_tiny_dynamic: the dynamic-frame recipe (speech_dataset_large.py) - natural-length utterances (61 / 150 / 225 mel frames), each
    log-mel on its own length, zero-padded mel frames attending freely in the encoder (reference quirk Q9), right padding only."""
    _step_vs_fixture(rf.load(name), small=True)


def test_cuda_step_matches_reference_run_at_real_widths():
    _step_vs_fixture(rf.load("ref_realwidth.pt"), small=False)
