"""Per-kernel numerics on the GPU: every C-ABI entry point against a plain PyTorch fp32 reference
of the same op on identical seeded inputs.  Tolerances are written next to each check (bf16 I/O,
fp32 accumulation)."""
import math

import pytest
import torch

pytestmark = pytest.mark.gpu

BF16, F32 = torch.bfloat16, torch.float32


@pytest.fixture(scope="module")
def ops():
    from slam_llm_b200 import ops as _ops
    return _ops


def dev():
    return torch.device("cuda:0")


def rnd(*shape, scale=1.0, dtype=BF16, seed=None):
    g = torch.Generator(device="cuda")
    g.manual_seed(1234 if seed is None else seed)
    return (torch.randn(*shape, device=dev(), generator=g, dtype=F32) * scale).to(dtype)


def rel_err(a, b):
    a, b = a.float(), b.float()
    return ((a - b).abs().max() / b.abs().max().clamp_min(1e-20)).item()


def cos_sim(a, b):
    a, b = a.float().flatten(), b.float().flatten()
    return torch.nn.functional.cosine_similarity(a, b, dim=0).item()


# ----------------------------------------------------------------------------------------------- GEMM
@pytest.mark.parametrize("M,N,K,bn", [
    (128, 256, 64, 256), (128, 128, 128, 128), (128, 64, 256, 64),
    (1600, 4096, 4096, 0), (300, 384, 1920, 0), (308, 2048, 512, 256),
    (1, 64, 64, 64), (257, 1280, 1280, 128), (1200, 6144, 4096, 256), (77, 5120, 240, 0),
    (1600, 4096, 4096, 192), (300, 200, 512, 192), (1600, 6144, 4096, 192),
    (1600, 4096, 4096, 256256), (1600, 4096, 6144, 256224), (6000, 1280, 1280, 256256), (129, 256, 64, 256256),
    # CTA-pair kernels (cta_group::2): 256 x BLOCK_N per SM pair
    (1604, 4096, 4096, 2000256), (6000, 1280, 1280, 2000224), (300, 384, 1920, 2000192), (257, 520, 640, 2000160), (129, 256, 64, 2000128), (1, 64, 64, 2000128),
])
def test_gemm_plain(ops, M, N, K, bn):
    a, b = rnd(M, K, seed=1), rnd(N, K, seed=2)
    out = ops.gemm(a, b, block_n=bn)
    ref = a.float() @ b.float().t()
    torch.cuda.synchronize()
    # bf16 output rounding (2^-9 relative) on |ref| up to ~sqrt(K)*4: compare relative to max
    assert rel_err(out, ref) < 6e-3, (M, N, K, bn, rel_err(out, ref))
    assert cos_sim(out, ref) > 0.9999


def test_gemm_f32_out_exactness(ops):
    # small integers: products and sums are exact in fp32, so the tcgen05 path must match bit-for-bit
    g = torch.Generator(device="cuda"); g.manual_seed(7)
    a = torch.randint(-4, 5, (300, 512), device=dev(), generator=g).to(BF16)
    b = torch.randint(-4, 5, (520, 512), device=dev(), generator=g).to(BF16)
    out = ops.gemm(a, b, out_f32=True)
    ref = a.float() @ b.float().t()
    assert torch.equal(out, ref)


@pytest.mark.parametrize("act", [0, 1, 2])
def test_gemm_epilogue(ops, act):
    M, N, K = 520, 1280, 640
    a, b = rnd(M, K, scale=0.5, seed=3), rnd(N, K, scale=0.1, seed=4)
    bias = rnd(N, dtype=F32, seed=5)
    res = rnd(M, N, seed=6)
    out = ops.gemm(a, b, bias=bias, residual=res, act=act, alpha=0.5, block_n=(0, 256256, 128192)[act])
    z = 0.5 * (a.float() @ b.float().t()) + bias
    if act == 1:
        z = torch.nn.functional.gelu(z)
    elif act == 2:
        z = torch.relu(z)
    ref = z + res.float()
    assert rel_err(out, ref) < 6e-3


@pytest.mark.parametrize("tile", [0, 128256, 128192, 256256, 2000256, 2000224])
def test_gemm_dual_segment_lora(ops, tile):
    # y = x W^T + (x A^T)(s B)^T accumulated in one TMEM tile
    M, N, K, R = 1600, 6144, 4096, 64
    x, w = rnd(M, K, seed=8), rnd(N, K, scale=0.02, seed=9)
    t, bs = rnd(M, R, seed=10), rnd(N, R, scale=0.05, seed=11)
    out = ops.gemm(x, w, a2=t, b2=bs, block_n=tile)
    ref = x.float() @ w.float().t() + t.float() @ bs.float().t()
    assert rel_err(out, ref) < 6e-3
    only_base = ops.gemm(x, w)
    assert rel_err(only_base, ref) > 2e-2  # the second segment really contributes


def _block64(w_gate, w_up):
    f, d = w_gate.shape
    return torch.stack([w_gate.view(f // 64, 64, d), w_up.view(f // 64, 64, d)], 1).reshape(2 * f, d).contiguous()


@pytest.mark.parametrize("M,F,K,tile", [(300, 512, 256, 0), (1604, 1792, 512, 128256), (1604, 1792, 512, 2000256), (77, 128, 64, 128128), (520, 1024, 320, 256256)])
def test_gemm_fused_swiglu(ops, M, F, K, tile):
    """act 3 / 4 (HF LlamaMLP gate/up -> silu * up, and its backward) against the unfused kernels on the blocked-64 layout:
    the epilogues compute from the bf16-rounded tensors, so the results are bit-identical."""
    x, wg, wu = rnd(M, K, seed=94), rnd(F, K, scale=0.1, seed=95), rnd(F, K, scale=0.1, seed=96)
    wgu = _block64(wg, wu)
    gu_ref = ops.gemm(x, wgu, block_n=tile, tail_split=-1)     # (the fused epilogues never split the tail: same summation order)
    h_ref = ops.swiglu_fwd(gu_ref, block=64)
    h = torch.empty(M, F, device=dev(), dtype=BF16)
    gu = ops.gemm(x, wgu, act=3, aux=h, block_n=tile)
    assert torch.equal(gu, gu_ref) and torch.equal(h, h_ref)
    # the blocked layout is a permutation of the HF [gate | up] layout
    g_hf = ops.gemm(x, torch.cat([wg, wu], 0).contiguous(), tail_split=-1)
    assert torch.equal(ops.swiglu_fwd(g_hf), h_ref)
    # backward: dh = dy @ W_down^T-like product [M, F], then d(gu)
    dy, wd = rnd(M, K, seed=97), rnd(F, K, scale=0.1, seed=98)
    dh = ops.gemm(dy, wd, block_n=tile if tile % 1000 != 0 else 0, tail_split=-1)
    dgu_ref = ops.swiglu_bwd(gu_ref, dh, block=64)
    dgu = ops.gemm(dy, wd, act=4, aux=gu_ref, block_n=tile if tile % 1000 != 0 else 0)
    assert torch.equal(dgu, dgu_ref)
    # and against torch autograd of silu(g) * u in fp32 (tolerance: bf16 inputs/outputs)
    gr = gu_ref.view(M, F // 64, 2, 64)[:, :, 0].reshape(M, F).float().requires_grad_(True)
    ur = gu_ref.view(M, F // 64, 2, 64)[:, :, 1].reshape(M, F).float().requires_grad_(True)
    (torch.nn.functional.silu(gr) * ur).backward(dh.float())
    got = dgu.view(M, F // 64, 2, 64)
    assert rel_err(got[:, :, 0].reshape(M, F), gr.grad) < 8e-3 and rel_err(got[:, :, 1].reshape(M, F), ur.grad) < 8e-3


@pytest.mark.parametrize("M,N,K,tile", [(1604, 4096, 4096, 128256), (1604, 6144, 4096, 128256), (308, 4096, 32064, 128256), (1604, 4096, 4096, 128192),
                                        (300, 776, 1280, 128128), (77, 264, 256, 128256)])
def test_gemm_tail_split(ops, M, N, K, tile):
    """Last partial wave cut into k-slices (partials exchanged through the workspace): same result as the plain schedule up to
    fp32 summation order, bit-identical from run to run, full epilogue applied."""
    a, b = rnd(M, K, seed=90), rnd(N, K, scale=0.05, seed=91)
    bias, res = rnd(N, seed=92).float(), rnd(M, N, seed=93)
    plain = ops.gemm(a, b, bias=bias, residual=res, act=1, block_n=tile, tail_split=-1)
    outs = [ops.gemm(a, b, bias=bias, residual=res, act=1, block_n=tile, tail_split=8) for _ in range(3)]
    ref = torch.nn.functional.gelu(a.float() @ b.float().t() + bias) + res.float()
    assert torch.equal(outs[0], outs[1]) and torch.equal(outs[1], outs[2])
    assert rel_err(outs[0], ref) < 6e-3 and rel_err(outs[0], plain.float()) < 6e-3
    out32 = ops.gemm(a, b, out_f32=True, block_n=tile, tail_split=8)
    assert rel_err(out32, a.float() @ b.float().t()) < 1e-4


@pytest.mark.parametrize("M,N,K,K2,split", [(1600, 64, 4096, 0, 8), (308, 4096, 12800, 0, 3), (1600, 64, 6144, 64, 5), (257, 512, 640, 0, 4)])
def test_gemm_split_k(ops, M, N, K, K2, split):
    a, b = rnd(M, K, seed=60), rnd(N, K, scale=0.05, seed=61)
    a2 = rnd(M, K2, seed=62) if K2 else None
    b2 = rnd(N, K2, scale=0.05, seed=63) if K2 else None
    out = ops.gemm(a, b, a2=a2, b2=b2, out_f32=True, split_k=split)
    ref = a.float() @ b.float().t() + (a2.float() @ b2.float().t() if K2 else 0)
    assert rel_err(out, ref) < 1e-4           # fp32 accumulation, only the summation order differs


def test_gemm_strided_views(ops):
    # operands / outputs that are column slices of wider buffers (fused QKV style)
    M, K = 384, 512
    big_a = rnd(M, 3 * K, seed=12)
    a = big_a[:, K:2 * K]
    b = rnd(256, K, seed=13)
    big_out = torch.zeros(M, 1024, device=dev(), dtype=BF16)
    ops.gemm(a, b, out=big_out[:, 512:768])
    ref = a.float() @ b.float().t()
    assert rel_err(big_out[:, 512:768], ref) < 6e-3
    assert big_out[:, :512].abs().max().item() == 0 and big_out[:, 768:].abs().max().item() == 0


def test_wgrad_thin(ops):
    M, P, Q = 1600, 16, 4096
    a_full = rnd(M, 64, seed=14)
    a = a_full[:, 16:32]
    b = rnd(M, Q, seed=15)
    out = torch.empty(P, Q, device=dev(), dtype=F32)
    ops.wgrad_thin(a, b, out, scale=2.0)
    ref = 2.0 * a.float().t() @ b.float()
    assert rel_err(out, ref) < 1e-4
    acc = out.clone()
    ops.wgrad_thin(a, b, acc, scale=2.0, accumulate=True)              # accumulate mode: C += product
    assert rel_err(acc, 2.0 * out) < 1e-5
    for (Mx, Px, Qx, ld) in ((1601, 8, 1024, 64), (333, 64, 6144, 64), (1600, 32, 520, 32), (70, 16, 4096, 16)):   # tensor-core path
        af = rnd(Mx, ld, seed=50)
        bx = rnd(Mx, Qx + 8, seed=51)[:, :Qx]
        o = torch.empty(Px, Qx, device=dev(), dtype=F32)
        ops.wgrad_thin(af[:, :Px], bx, o, scale=0.5)
        assert rel_err(o, 0.5 * af[:, :Px].float().t() @ bx.float()) < 1e-4, (Mx, Px, Qx)
    out2 = torch.empty(40, 300, device=dev(), dtype=F32)
    a2, b2 = rnd(77, 40, seed=16), rnd(77, 300, seed=17)
    ops.wgrad_thin(a2, b2, out2)
    assert rel_err(out2, a2.float().t() @ b2.float()) < 1e-4


# ----------------------------------------------------------------------------------------------- front end
def _mel_filters(n_mels):
    from slam_llm_b200.frontend import mel_filterbank
    return mel_filterbank(n_mels).to(dev())


def _ref_logmel(wav, filters):
    window = torch.hann_window(400, device=wav.device)
    stft = torch.stft(wav, 400, 160, window=window, return_complex=True)
    mag = stft[..., :-1].abs() ** 2
    mel = filters @ mag
    lg = torch.clamp(mel, min=1e-10).log10()
    lg = torch.maximum(lg, lg.amax(dim=(-2, -1), keepdim=True) - 8.0)
    return ((lg + 4.0) / 4.0).permute(0, 2, 1).contiguous()


@pytest.mark.parametrize("n_mels,n_samples", [(80, 480000), (128, 480000), (80, 80000), (128, 16123)])
def test_logmel(ops, n_mels, n_samples):
    wav = rnd(3, n_samples, scale=0.1, dtype=F32, seed=18)
    wav[1, n_samples // 2:] = 0.0  # a zero-padded utterance (pad_or_trim)
    filt = _mel_filters(n_mels)
    out = ops.logmel(wav, filt.t().contiguous())
    ref = _ref_logmel(wav.double(), filt.double()).float()
    assert out.shape == ref.shape
    # fp32 direct DFT vs fp64 FFT reference, after log compression: absolute tolerance on the (x+4)/4 scale
    assert (out - ref).abs().max().item() < 2e-3, (out - ref).abs().max().item()


def test_logmel_variable_lengths(ops):
    """Dynamic-frame batches: each utterance is transformed on ITS OWN length and the mel (not the audio) is zero padded."""
    n_mels, n_max = 80, 40000
    lens = [40000, 23456, 16000]
    wav = rnd(3, n_max, scale=0.1, dtype=F32, seed=77)
    for i, n in enumerate(lens):
        wav[i, n:] = 0.0
    filt = _mel_filters(n_mels)
    out = ops.logmel(wav, filt.t().contiguous(), lengths=torch.tensor(lens, dtype=torch.int32, device=dev()))
    assert out.shape == (3, n_max // 160, n_mels)
    for i, n in enumerate(lens):
        ref = _ref_logmel(wav[i:i + 1, :n].double(), filt.double()).float()[0]      # [n//160, n_mels]
        assert (out[i, : n // 160] - ref).abs().max().item() < 2e-3
        if n // 160 < n_max // 160:
            assert out[i, n // 160:].abs().max().item() == 0.0


def test_conv_stem_im2col(ops):
    B, T, Cin, Cout = 2, 200, 80, 384
    x = rnd(B, T, Cin, dtype=F32, seed=19)
    w1 = rnd(Cout, Cin, 3, scale=0.1, dtype=F32, seed=20)
    b1 = rnd(Cout, dtype=F32, seed=21)
    ldk = 256  # 3*80 = 240 padded to a multiple of 8 (here 64)
    col = ops.conv_im2col(x, 1, ldk)
    wk = torch.zeros(Cout, ldk, device=dev(), dtype=BF16)
    wk[:, :3 * Cin] = w1.permute(0, 2, 1).reshape(Cout, 3 * Cin).to(BF16)
    y = ops.gemm(col, wk, bias=b1, act=1)
    ref = torch.nn.functional.gelu(torch.nn.functional.conv1d(x.permute(0, 2, 1), w1, b1, padding=1)).permute(0, 2, 1)
    assert rel_err(y.view(B, T, Cout), ref) < 1.5e-2
    # stride 2 on bf16 input
    x2 = y.view(B, T, Cout)
    w2 = rnd(Cout, Cout, 3, scale=0.05, dtype=F32, seed=22)
    col2 = ops.conv_im2col(x2, 2, 3 * Cout)
    y2 = ops.gemm(col2, w2.permute(0, 2, 1).reshape(Cout, 3 * Cout).to(BF16))
    ref2 = torch.nn.functional.conv1d(x2.float().permute(0, 2, 1), w2, None, stride=2, padding=1).permute(0, 2, 1)
    assert y2.shape[0] == B * 100
    assert rel_err(y2.view(B, 100, Cout), ref2) < 1.5e-2
    pos = rnd(150, Cout, dtype=F32, seed=23)
    y3 = ops.add_pos_(y2.view(B, 100, Cout).clone(), pos)
    assert rel_err(y3, y2.view(B, 100, Cout).float() + pos[:100]) < 1e-2


@pytest.mark.parametrize("d", [384, 512, 768, 1024, 1280])
def test_layernorm(ops, d):
    x = rnd(777, d, scale=2.0, seed=24)
    w, b = rnd(d, dtype=F32, seed=25), rnd(d, dtype=F32, seed=26)
    y = ops.layernorm(x, w, b)
    ref = torch.nn.functional.layer_norm(x.float(), (d,), w, b, 1e-5)
    assert rel_err(y, ref) < 8e-3


# ----------------------------------------------------------------------------------------------- attention
def _ref_attn(q, k, v, causal, scale, key_mask):
    # q [B,S,H,dh] ; fp32 math with explicit masking, GQA via repeat
    B, Sq, Hq, dh = q.shape
    Hkv = k.shape[2]
    qf, kf, vf = q.float().transpose(1, 2), k.float().transpose(1, 2), v.float().transpose(1, 2)
    kf = kf.repeat_interleave(Hq // Hkv, dim=1)
    vf = vf.repeat_interleave(Hq // Hkv, dim=1)
    s = qf @ kf.transpose(-1, -2) * scale
    mask = torch.ones(B, 1, Sq, k.shape[1], dtype=torch.bool, device=q.device)
    if causal:
        mask = mask & torch.ones(Sq, Sq, dtype=torch.bool, device=q.device).tril()
    if key_mask is not None:
        mask = mask & key_mask.bool()[:, None, None, :]
    s = s.masked_fill(~mask, float("-inf"))
    p = torch.softmax(s, dim=-1)
    p = torch.nan_to_num(p, nan=0.0)
    return (p @ vf).transpose(1, 2)


@pytest.mark.parametrize("B,S,Hq,Hkv,dh,causal,masked", [
    (2, 1500, 6, 6, 64, False, False),     # whisper-tiny encoder
    (1, 333, 20, 20, 64, False, False),    # ragged length
    (2, 400, 32, 8, 128, True, True),      # Llama-3-8B decoder, GQA 4:1
    (2, 150, 32, 4, 64, True, True),       # TinyLlama decoder, GQA 8:1
    (1, 65, 4, 4, 128, True, False),
    (4, 401, 32, 8, 128, True, True),      # BASELINE config 3 decoder shape (tcgen05 kernel, dh = 128)
    (1, 700, 8, 8, 128, True, False),      # several key tiles, causal tile skipping
    (2, 200, 4, 4, 64, False, True),       # key mask without causal
    (1, 40, 4, 2, 64, True, True),         # short: mma.sync kernel
    # tile and dispatch edges (tcgen05 from S = 64, 128-key / 128-query tiles; mma.sync below): with B = 3 the 128-row TMA tiles of
    # samples 0 and 1 reach into the next sample's rows
    *[(3, S, 8, 2, 128, True, True) for S in (63, 64, 127, 128, 129, 255, 257)],
    *[(3, S, 4, 4, 64, False, False) for S in (63, 64, 127, 128, 129, 255, 257)],
])
def test_attention_fwd_bwd(ops, B, S, Hq, Hkv, dh, causal, masked):
    qkv = rnd(B * S, (Hq + 2 * Hkv) * dh, seed=27)  # fused QKV buffer, used in place
    q = qkv[:, :Hq * dh].view(B, S, Hq, dh)
    k = qkv[:, Hq * dh:(Hq + Hkv) * dh].view(B, S, Hkv, dh)
    v = qkv[:, (Hq + Hkv) * dh:].view(B, S, Hkv, dh)
    key_mask = None
    if masked:
        key_mask = torch.ones(B, S, dtype=torch.uint8, device=dev())
        key_mask[0, :7] = 0          # left padding on sample 0
        key_mask[-1, S - 5:] = 0     # right padding on the last sample
    scale = 1.0 / math.sqrt(dh)
    out, lse = ops.attn_fwd(q, k, v, causal=causal, scale=scale, key_mask=key_mask, need_lse=True)
    qr, kr, vr = (t.detach().float().requires_grad_(True) for t in (q, k, v))
    ref = _ref_attn(qr, kr, vr, causal, scale, key_mask)
    valid = torch.ones(B, S, dtype=torch.bool, device=dev()) if key_mask is None else key_mask.bool()
    sel = valid[:, :, None, None].expand_as(ref)
    assert rel_err(out[sel], ref[sel]) < 1.5e-2, rel_err(out[sel], ref[sel])
    # lse [B, Hq, S] (natural log) against the fp32 logsumexp of the masked scores, on rows that see at least one key
    sc = (qr.detach().transpose(1, 2) @ kr.detach().transpose(1, 2).repeat_interleave(Hq // Hkv, dim=1).transpose(-1, -2)) * scale
    m = torch.ones(B, 1, S, S, dtype=torch.bool, device=dev())
    if causal:
        m = m & torch.ones(S, S, dtype=torch.bool, device=dev()).tril()
    if key_mask is not None:
        m = m & key_mask.bool()[:, None, None, :]
    lse_ref = torch.logsumexp(sc.masked_fill(~m, float("-inf")), dim=-1)
    ok = torch.isfinite(lse_ref)
    assert (lse[ok] - lse_ref[ok]).abs().max().item() < 2e-2, (lse[ok] - lse_ref[ok]).abs().max().item()
    if not causal:
        return
    dout = rnd(B, S, Hq, dh, seed=28) * valid[:, :, None, None].to(BF16)  # padded query rows get zero grad
    dq, dk, dv = ops.attn_bwd(q, k, v, out, lse, dout, causal=causal, scale=scale, key_mask=key_mask)
    ref.backward(dout.float())
    for got, want, name in ((dq, qr.grad, "dq"), (dk, kr.grad, "dk"), (dv, vr.grad, "dv")):
        assert rel_err(got, want) < 3e-2, (name, rel_err(got, want))
        assert cos_sim(got, want) > 0.999, (name, cos_sim(got, want))
    # rope=(cos, sin): the finishing kernel also applies the inverse rotation to dQ / dK (gradients w.r.t. the un-rotated projections)
    cos, sin = _rope_tables(S, dh, 500000.0)
    dq2, dk2, dv2 = ops.attn_bwd(q, k, v, out, lse, dout, causal=causal, scale=scale, key_mask=key_mask, rope=(cos, sin))

    def unrotate(g):
        c = torch.cat([cos, cos], -1)[None, :, None, :]
        s_ = torch.cat([sin, sin], -1)[None, :, None, :]
        g = g.float()
        rot = torch.cat([g[..., dh // 2:], -g[..., :dh // 2]], -1)          # R^T g = g cos - rotate_half(g) sin
        return g * c + rot * s_
    assert rel_err(dq2, unrotate(qr.grad)) < 3e-2 and cos_sim(dq2, unrotate(qr.grad)) > 0.999
    assert rel_err(dk2, unrotate(kr.grad)) < 3e-2 and cos_sim(dk2, unrotate(kr.grad)) > 0.999
    assert rel_err(dv2, vr.grad) < 3e-2


@pytest.mark.parametrize("B,S,H", [(2, 1500, 6), (1, 333, 20), (4, 1500, 20), (3, 128, 2), (1, 129, 1), (2, 1000, 8)])
def test_attention_encoder_tcgen05(ops, B, S, H):
    """Whisper-encoder shape (dh = 64, non-causal, unmasked, no lse): served by the tcgen05/TMEM kernel (fmha_tc.cu)."""
    d = H * 64
    qkv = rnd(B * S, 3 * d, seed=70)
    q, k, v = (qkv[:, i * d:(i + 1) * d].view(B, S, H, 64) for i in range(3))
    out, _ = ops.attn_fwd(q, k, v, causal=False, scale=0.125)
    ref = _ref_attn(q, k, v, False, 0.125, None)
    assert rel_err(out, ref) < 1.5e-2, rel_err(out, ref)
    assert cos_sim(out, ref) > 0.9995


# ----------------------------------------------------------------------------------------------- merge
def _ref_merge(ids, mask, audio, embed):
    ids = ids.clone()
    ids[ids == -1] = 0
    emb = embed.float()[ids]
    start = (mask == 1).float().argmax(dim=1)
    lens = torch.clamp(mask.sum(dim=1), max=audio.shape[1]).tolist()
    pad = torch.zeros_like(emb)
    for i in range(audio.shape[0]):
        pad[i, start[i]:start[i] + lens[i]] = audio[i, :lens[i]].float()
    return pad + emb * (~mask.bool())[:, :, None]


def test_embed_merge(ops):
    B, S, Ta, D, V = 3, 50, 12, 256, 1000
    g = torch.Generator(device="cuda"); g.manual_seed(3)
    ids = torch.randint(0, V, (B, S), device=dev(), generator=g)
    mask = torch.zeros(B, S, dtype=torch.uint8, device=dev())
    mask[0, 0:12] = 1; ids[0, 0:12] = -1
    mask[1, 5:15] = 1; ids[1, 5:15] = -1       # shorter than Ta
    mask[2, 3:23] = 1; ids[2, 3:23] = -1       # longer than Ta: clamp
    audio, embed = rnd(B, Ta, D, seed=29), rnd(V, D, seed=30)
    x = ops.embed_merge(ids, mask, audio, embed)
    ref = _ref_merge(ids, mask, audio, embed)
    assert torch.equal(x.float(), ref)         # pure data movement: exact
    dx = rnd(B, S, D, seed=31)
    da = ops.embed_merge_bwd(mask, dx, Ta)
    a_leaf = audio.float().requires_grad_(True)
    _ref_merge(ids, mask, a_leaf, embed).backward(dx.float())
    assert torch.equal(da.float(), a_leaf.grad)


# ----------------------------------------------------------------------------------------------- decoder element-wise
@pytest.mark.parametrize("d", [2048, 4096, 896, 1024, 512])
def test_rmsnorm(ops, d):
    x, w = rnd(333, d, scale=3.0, seed=32), (rnd(d, seed=33) * 0.1 + 1.0).to(BF16)
    y, rstd = ops.rmsnorm_fwd(x, w, 1e-5)
    xr = x.float().requires_grad_(True)
    ref = xr * torch.rsqrt(xr.pow(2).mean(-1, keepdim=True) + 1e-5) * w.float()
    assert rel_err(y, ref) < 8e-3
    dy, dres = rnd(333, d, seed=34), rnd(333, d, seed=35)
    dx = ops.rmsnorm_bwd(dy, x, w, rstd, dres)
    ref.backward(dy.float())
    assert rel_err(dx, xr.grad + dres.float()) < 8e-3


@pytest.mark.parametrize("tile", [0, 2000192, 2000224, 2000256, 128192, 128128, 4000192])
def test_gemm_transpose_out_swap_ab(ops, tile):
    """transpose_out: the WEIGHT is the M operand (CTA-pair tiles without row padding), tokens are the N operand; the result still lands as
    y[tokens, features] = x W^T + x2 W2^T + residual.  Integer-valued inputs: exact in fp32 accumulation -> bit-exact after bf16 rounding."""
    Mx, Nw, K, r = 1604, 768, 320, 64                     # (768 weight rows: the 512-row tiles of 4000192 run half empty in their second row block)
    g = torch.Generator(device="cuda").manual_seed(91)
    x = torch.randint(-3, 4, (Mx, K), generator=g, device="cuda").to(BF16)
    w = torch.randint(-3, 4, (Nw, K), generator=g, device="cuda").to(BF16)
    x2 = torch.randint(-2, 3, (Mx, r), generator=g, device="cuda").to(BF16)
    w2 = torch.randint(-2, 3, (Nw, r), generator=g, device="cuda").to(BF16)
    res = torch.randint(-8, 9, (Mx, Nw), generator=g, device="cuda").to(BF16)
    want = x.float() @ w.float().t()
    y = ops.gemm(w, x, transpose_out=True, block_n=tile)
    assert y.shape == (Mx, Nw) and torch.equal(y.float(), want.to(BF16).float())
    want2 = want + x2.float() @ w2.float().t() + res.float()
    y2 = ops.gemm(w, x, a2=w2, b2=x2, residual=res, transpose_out=True, block_n=tile)
    assert torch.equal(y2.float(), want2.to(BF16).float())
    # in-place residual (out aliases residual), as the decoder's o / down projections use it
    buf = res.clone()
    ops.gemm(w, x, residual=buf, out=buf, transpose_out=True, block_n=tile)
    assert torch.equal(buf.float(), (want + res.float()).to(BF16).float())
    # strided output rows (a column slice of a wider buffer)
    wide = torch.zeros(Mx, Nw + 64, device="cuda", dtype=BF16)
    ops.gemm(w, x, out=wide[:, 32: 32 + Nw], transpose_out=True, block_n=tile)
    assert torch.equal(wide[:, 32: 32 + Nw].float(), want.to(BF16).float()) and float(wide[:, :32].abs().max()) == 0.0


@pytest.mark.parametrize("shape", [(1604, 64, 4096), (1604, 64, 6144), (300, 16, 1032), (128, 64, 14336), (4, 64, 4096), (1604, 40, 1024)])
def test_gemm_thin_cluster(ops, shape):
    """Thin products (N <= 64): a cluster of 8 CTAs per 128-row tile splits K and reduces the partial tiles through distributed shared memory
    in rank order (csrc/gemm_thin.cuh).  Integer-valued inputs: exact in fp32 -> bit-exact after the bf16 rounding; `auto` must pick the
    cluster kernel for these shapes and agree with the explicit choice and with the one-CTA-per-tile kernel."""
    M, N, K = shape
    g = torch.Generator(device="cuda").manual_seed(17 + M + K)
    a = torch.randint(-3, 4, (M, K), generator=g, device="cuda").to(BF16)
    b = torch.randint(-3, 4, (N, K), generator=g, device="cuda").to(BF16)
    want = (a.float() @ b.float().t() * 0.5).to(BF16)
    y = ops.gemm(a, b, alpha=0.5, block_n=3000064)
    assert y.shape == (M, N) and torch.equal(y, want)
    assert torch.equal(ops.gemm(a, b, alpha=0.5), want)                      # auto
    assert torch.equal(ops.gemm(a, b, alpha=0.5, block_n=64), want)          # the 128 x 64 one-CTA kernel
    # real-valued inputs: deterministic (fixed reduction order) and within bf16 rounding of the fp32 product
    a, b = rnd(M, K, seed=5), rnd(N, K, seed=6)
    y1, y2 = ops.gemm(a, b, block_n=3000064), ops.gemm(a, b, block_n=3000064)
    assert torch.equal(y1, y2)
    ref = a.float() @ b.float().t()
    assert float((y1.float() - ref).abs().max()) <= 0.01 * float(ref.abs().max()) + 1e-3
    # a row-strided output (the LoRA products are written into slices of wider buffers)
    wide = torch.zeros(M, N + 16, device="cuda", dtype=BF16)
    ops.gemm(a, b, out=wide[:, 8: 8 + N], block_n=3000064)
    assert torch.equal(wide[:, 8: 8 + N], y1) and float(wide[:, :8].abs().max()) == 0.0 and float(wide[:, 8 + N:].abs().max()) == 0.0


@pytest.mark.parametrize("M,F,K,tile", [(1604, 1792, 512, 0), (1604, 1792, 512, 2000256), (300, 512, 256, 2000192), (77, 128, 64, 2000160)])
def test_gemm_fused_swiglu_bwd_swapped(ops, M, F, K, tile):
    """act 4 with transpose_out (swap-AB d_down): W_down^T [F, K] is the M operand, dY [M, K] the N operand, gate / up and d(gu) are read / written
    transposed through the epilogue's staging tile.  Same k order and the same per-element math as the non-swapped fused kernel: bit-identical."""
    x, wg, wu = rnd(M, K, seed=194), rnd(F, K, scale=0.1, seed=195), rnd(F, K, scale=0.1, seed=196)
    gu = ops.gemm(x, _block64(wg, wu), tail_split=-1)
    dy, wd = rnd(M, K, seed=197), rnd(F, K, scale=0.1, seed=198)
    want = ops.gemm(dy, wd, act=4, aux=gu, block_n=2000256)
    got = ops.gemm(wd, dy, act=4, aux=gu, transpose_out=True, block_n=tile, static_w=True)
    assert got.shape == (M, 2 * F) and torch.equal(got, want)
    assert torch.equal(got, ops.swiglu_bwd(gu, ops.gemm(dy, wd, tail_split=-1), block=64))     # and to the unfused pair of kernels


def test_gemm_pair512_single_round(ops):
    """Tile 4000192 ("pair512": 512 x 192 per SM pair, one accumulator set) on the shape it is used for - 4096 weight rows x 1604 tokens = 72 tiles,
    one round - with a long K, the LoRA segment and the residual; bit-exact on integer-valued inputs, equal to the 256-row schedule otherwise."""
    Mx, Nw, K, r = 1604, 4096, 2048, 64
    g = torch.Generator(device="cuda").manual_seed(123)
    x = torch.randint(-2, 3, (Mx, K), generator=g, device="cuda").to(BF16)
    w = torch.randint(-2, 3, (Nw, K), generator=g, device="cuda").to(BF16)
    x2 = torch.randint(-2, 3, (Mx, r), generator=g, device="cuda").to(BF16)
    w2 = torch.randint(-2, 3, (Nw, r), generator=g, device="cuda").to(BF16)
    res = torch.randint(-8, 9, (Mx, Nw), generator=g, device="cuda").to(BF16)
    want = (x.float() @ w.float().t() + x2.float() @ w2.float().t() + res.float()).to(BF16)
    y = ops.gemm(w, x, a2=w2, b2=x2, residual=res, transpose_out=True, block_n=4000192, static_w=True)
    assert torch.equal(y, want)
    xr, wr = rnd(Mx, K, seed=31), rnd(Nw, K, scale=0.05, seed=32)
    a = ops.gemm(wr, xr, residual=res, transpose_out=True, block_n=4000192)
    b = ops.gemm(wr, xr, residual=res, transpose_out=True, block_n=2000192)
    assert torch.equal(a, b)                                 # same k order per output element: identical fp32 accumulation
    # several tiles per pair (no accumulator double buffering: the MMA waits for the epilogue): 8192 weight rows = 144 tiles on 74 pairs
    w8 = torch.randint(-2, 3, (8192, 256), generator=g, device="cuda").to(BF16)
    x8 = torch.randint(-2, 3, (Mx, 256), generator=g, device="cuda").to(BF16)
    assert torch.equal(ops.gemm(w8, x8, transpose_out=True, block_n=4000192), (x8.float() @ w8.float().t()).to(BF16))


def _rope_tables(S, dh, theta):
    inv = 1.0 / (theta ** (torch.arange(0, dh, 2, dtype=F32, device=dev()) / dh))
    fr = torch.outer(torch.arange(S, dtype=F32, device=dev()), inv)
    return fr.cos().contiguous(), fr.sin().contiguous()


def test_rope(ops):
    B, S, H, dh = 2, 100, 8, 128
    buf = rnd(B * S, 3 * H * dh, seed=36)
    x = buf[:, H * dh:2 * H * dh]
    x0 = x.clone()
    cos, sin = _rope_tables(S, dh, 500000.0)
    ops.rope_(x, H, dh, S, cos, sin)
    xf = x0.float().view(B, S, H, dh)
    c = torch.cat([cos, cos], -1)[None, :, None, :]
    s = torch.cat([sin, sin], -1)[None, :, None, :]
    rot = torch.cat([-xf[..., dh // 2:], xf[..., :dh // 2]], -1)
    ref = xf * c + rot * s
    assert rel_err(x.reshape(B, S, H, dh), ref) < 8e-3
    assert torch.equal(buf[:, :H * dh], rnd(B * S, 3 * H * dh, seed=36)[:, :H * dh])  # neighbours untouched
    ops.rope_(x, H, dh, S, cos, sin, inverse=True)
    assert rel_err(x, x0) < 1.2e-2  # rotation then inverse rotation (two bf16 roundings)


def test_swiglu(ops):
    rows, f = 257, 1408
    gu = rnd(rows, 2 * f, scale=2.0, seed=37)
    h = ops.swiglu_fwd(gu)
    gr = gu.float().requires_grad_(True)
    ref = torch.nn.functional.silu(gr[:, :f]) * gr[:, f:]
    assert rel_err(h, ref) < 8e-3
    dh_ = rnd(rows, f, seed=38)
    dgu = ops.swiglu_bwd(gu, dh_)
    ref.backward(dh_.float())
    assert rel_err(dgu, gr.grad) < 8e-3


# ----------------------------------------------------------------------------------------------- loss / optimizer
@pytest.mark.parametrize("V", [32000, 128256, 1000])
def test_cross_entropy(ops, V):
    R = 37
    logits = rnd(R, V, scale=3.0, dtype=F32, seed=39)
    g = torch.Generator(device="cuda"); g.manual_seed(5)
    tgt = torch.randint(0, V, (R,), device=dev(), generator=g)
    tgt[3] = -100; tgt[10] = -100
    for r in (0, 5, 20):
        tgt[r] = logits[r].argmax()
    stats = (torch.zeros(1, device=dev()), torch.zeros(1, dtype=torch.int32, device=dev()), torch.zeros(1, dtype=torch.int32, device=dev()))
    gs = torch.tensor([1.0 / 35], device=dev())
    dl = torch.empty(R, V, device=dev(), dtype=BF16)
    ops.cross_entropy(logits, tgt, stats, dl, gs)
    lr = logits.clone().requires_grad_(True)
    ref_loss = torch.nn.functional.cross_entropy(lr, tgt, ignore_index=-100, reduction="sum")
    assert abs(stats[0].item() - ref_loss.item()) / ref_loss.item() < 1e-5
    assert stats[1].item() == 35
    valid = tgt != -100
    assert stats[2].item() == (logits.argmax(-1)[valid] == tgt[valid]).sum().item()
    (ref_loss / 35).backward()
    assert (dl.float() - lr.grad).abs().max().item() < 2e-4  # bf16 rounding of probabilities / 35
    assert dl[3].abs().max().item() == 0


def test_adamw(ops):
    n = 100003
    p0, g0 = rnd(n, dtype=F32, seed=40), rnd(n, dtype=F32, seed=41)
    p = p0.clone(); m = torch.zeros_like(p); v = torch.zeros_like(p)
    pr = torch.nn.Parameter(p0.clone())
    opt = torch.optim.AdamW([pr], lr=1e-3, weight_decay=0.01)
    for step in range(1, 4):
        g = g0 * step
        ops.adamw_(p, g * 2.0, m, v, lr=1e-3, weight_decay=0.01, step=step, grad_div=2.0)
        pr.grad = g.clone()
        opt.step()
    assert (p - pr.data).abs().max().item() < 2e-6


# ----------------------------------------------------------------------------------------------- utilities
def test_utilities(ops):
    x = rnd(513, 300, dtype=F32, seed=42)
    xb = ops.cast_bf16(x, scale=0.5)
    assert torch.equal(xb, (x * 0.5).to(BF16))
    assert torch.equal(ops.cast_f32(xb), xb.float())
    xt = ops.transpose(xb)
    assert torch.equal(xt, xb.t().contiguous())
    xw = rnd(100, 256, seed=43)
    idx = torch.tensor([5, 99, 0, 42], dtype=torch.int32, device=dev())
    gth = ops.gather_rows(xw, idx)
    assert torch.equal(gth, xw[idx.long()])
    dst = torch.zeros_like(xw)
    ops.scatter_rows(gth, idx, dst)
    assert torch.equal(dst[idx.long()], gth)
    y = rnd(300, 200, seed=44)
    dy = rnd(300, 200, seed=45)
    assert torch.equal(ops.relu_bwd(dy, y), torch.where(y.float() > 0, dy, torch.zeros_like(dy)))
    cs = torch.empty(200, device=dev(), dtype=F32)
    ops.colsum(y, cs)
    assert rel_err(cs, y.float().sum(0)) < 1e-5
    assert torch.equal(ops.add(y, dy), (y.float() + dy.float()).to(BF16))
    # pack2d: batched strided cast with and without transpose
    src = rnd(3, 16, 40, dtype=F32, seed=46)
    dst = torch.zeros(3, 64, 40, device=dev(), dtype=BF16)
    ops.pack2d(src, dst, batch=3, rows=16, cols=40, src_bs=16 * 40, src_ld=40, dst_bs=64 * 40, dst_ld=40, dst_off=16 * 40, scale=2.0)
    assert torch.equal(dst[:, 16:32], (src * 2.0).to(BF16)) and dst[:, :16].abs().max().item() == 0
    dstt = torch.zeros(3, 40, 64, device=dev(), dtype=BF16)
    ops.pack2d(src, dstt, batch=3, rows=16, cols=40, src_bs=16 * 40, src_ld=40, dst_bs=40 * 64, dst_ld=64, dst_off=32, transpose=True)
    assert torch.equal(dstt[:, :, 32:48], src.transpose(1, 2).to(BF16))


# ----------------------------------------------------------------------------------------------- full fine-tune reductions (fp64 references)
# The kernels below sum fp32 terms in a fixed tree: a run of terms per thread, 8 row lanes, then one fp32 atomic per row slice (at most 64).
# Whatever the order, the rounding error of an n-term fp32 sum is at most about n * 2^-24 * sum|terms| (recursive summation bound); every
# path here has n < 170, so |err| <= 1e-5 * sum|terms| holds with margin.
SUM_BOUND = 1e-5


@pytest.mark.parametrize("rows", [1, 257, 1604, 16400])
@pytest.mark.parametrize("d", [896, 900, 4096])
def test_rmsnorm_wgrad(ops, rows, d):
    """dw[c] += sum_r dy[r,c] * x[r,c] * rstd[r], accumulated into a non-zero dw; 16400 rows use the 64-way row split."""
    dy, x = rnd(rows, d, seed=110), rnd(rows, d, scale=2.0, seed=111)
    g = torch.Generator(device="cuda").manual_seed(112)
    rstd = torch.rand(rows, device=dev(), generator=g) * 1.5 + 0.5
    dw0 = rnd(d, dtype=F32, seed=113)
    dw = ops.rmsnorm_wgrad(dy, x, rstd, dw0.clone())
    terms = dy.double() * x.double() * rstd.double()[:, None]
    ref = dw0.double() + terms.sum(0)
    bound = SUM_BOUND * (dw0.double().abs() + terms.abs().sum(0))
    assert ((dw.double() - ref).abs() <= bound).all(), ((dw.double() - ref).abs() / bound).max().item()


def test_embed_grad(ops):
    """dE[max(id, 0)] += dx[r] for text rows (modality mask 0): repeated ids accumulate, -1 goes to row 0, ids >= vocab and audio rows are
    skipped.  Rows nobody writes keep their value bit for bit; the guard rows after the table are never written."""
    V, d, rows = 1000, 896, 300
    g = torch.Generator(device="cuda").manual_seed(120)
    ids = torch.randint(0, 40, (rows,), device=dev(), generator=g)        # 40 distinct ids over 300 rows: many repeats
    ids[::7] = -1
    ids[5::11] = V + 3
    ids[6] = V
    mask = torch.zeros(rows, dtype=torch.uint8, device=dev())
    mask[100:160] = 1
    dx = rnd(rows, d, seed=121)
    table = torch.full((V + 8, d), float("nan"), device=dev(), dtype=F32)
    table[:V] = rnd(V, d, dtype=F32, seed=122)
    de0 = table[:V].clone()
    ops.embed_grad(ids, mask, dx, table[:V])
    keep = (mask == 0) & (ids < V)
    tgt = ids.clamp_min(0)[keep]
    ref, absum = de0.double(), de0.double().abs()
    ref.index_add_(0, tgt, dx.double()[keep])
    absum.index_add_(0, tgt, dx.double().abs()[keep])
    assert ((table[:V].double() - ref).abs() <= SUM_BOUND * absum).all()
    untouched = torch.ones(V, dtype=torch.bool, device=dev())
    untouched[tgt] = False
    assert torch.equal(table[:V][untouched], de0[untouched])
    assert torch.isnan(table[V:]).all()


@pytest.mark.parametrize("batch,rows,cols", [(3, 45, 77), (2, 100, 33), (1, 31, 1), (4, 64, 96)])
def test_transpose_f32_batched(ops, batch, rows, cols):
    """dst[b][j][i] = src[b][i][j], sides not multiples of the 32 x 32 tile: pure data movement, exact; every element written."""
    src = rnd(batch, rows, cols, dtype=F32, seed=130)
    dst = torch.full((batch, cols, rows), float("nan"), device=dev(), dtype=F32)
    ops.transpose_f32_batched(src, dst, batch, rows, cols)
    assert torch.equal(dst, src.transpose(1, 2))


@pytest.mark.parametrize("rows,cols", [(6007, 200), (20000, 1000), (1, 72)])
def test_colsum(ops, rows, cols):
    """out[c] = sum_r x[r,c] on a column slice of a wider buffer (row stride != cols) into a NaN-filled out: the kernel zeroes it first;
    20000 rows use the 64-way row split."""
    big = rnd(rows, cols + 24, scale=3.0, seed=140)
    x = big[:, 8:8 + cols]
    out = torch.full((cols,), float("nan"), device=dev(), dtype=F32)
    ops.colsum(x, out)
    ref = x.double().sum(0)
    assert ((out.double() - ref).abs() <= SUM_BOUND * x.double().abs().sum(0)).all()
