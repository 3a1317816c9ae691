"""Attention kernels (tcgen05 flash kernels in fmha_tc.cu, mma.sync kernels in attention.cu, the shared finishing kernel) against a plain
fp64 reference at the inputs where flash attention goes wrong: large and rising logits, long padding and query rows that see no key,
masked keys holding large values, decode shapes (Sq != Sk), GQA group 7 and the production gradient layout.

Errors are measured per query row (per key row for dK / dV) and per (sample, head), not per tensor, so an error confined to one sample,
one head or the tail tile cannot hide below the largest value elsewhere.
"""
import math

import pytest
import torch

pytestmark = pytest.mark.gpu

BF16, F32 = torch.bfloat16, torch.float32

# Forward output, per query row: max|got - ref| over the row / max|ref| over the row, where a row far smaller than the largest row of its
# (sample, head) is measured against 1/64 of that row.  Tolerance: P rounded to bf16 before P V (2^-9 relative per term) plus the bf16
# rounding of the output (2^-9); measured <= 7.1e-3 on a B200.
OUT_FLOOR, TOL_OUT = 1.0 / 64, 1.0e-2
# dQ / dK / dV, per query (dQ) or key (dK, dV) row: max|got - ref| over the row / max|ref| over its (sample, head).  A gradient row whose terms
# cancel keeps the rounding of the terms, not of the result: P and dS = P (dP - delta) are rounded to bf16 before the gradient MMAs and
# delta comes from the bf16 forward output, so the error scales with the (sample, head), not with the row.  Measured <= 9.2e-3 on a B200
# (the large-logit case has its own bound below).
GRAD_FLOOR, TOL_GRAD = 1.0, 1.5e-2
# A (sample, head) whose exact gradient vanishes (every query sees at most one key: a one-element softmax has no gradient) still gets the
# fp32 rounding of dP - delta: every row is also measured against at least 1e-3 of the largest row of the whole tensor.
TENSOR_FLOOR = 1.0e-3
# Cosine per (sample, head): the roundings above are independent from element to element (measured >= 0.99996).
COS_MIN = 0.9999
# lse: scores accumulate in fp32 from bf16 q / k, the row sum stays in fp32 (no bf16 rounding), ex2.approx adds 2^-22 relative:
# an absolute term for |lse| ~ 1 plus a relative term for the large-logit rows (|lse| up to ~100).
LSE_ABS, LSE_REL = 2.0e-4, 2.0e-5


def dev():
    return torch.device("cuda:0")


def gen(seed):
    g = torch.Generator(device="cuda")
    g.manual_seed(seed)
    return g


def randn(*shape, seed, scale=1.0):
    return torch.randn(*shape, device=dev(), generator=gen(seed), dtype=F32) * scale


def rope_tables(S, dh, theta=500000.0):
    inv = 1.0 / (theta ** (torch.arange(0, dh, 2, dtype=F32, device=dev()) / dh))
    fr = torch.outer(torch.arange(S, dtype=F32, device=dev()), inv)
    return fr.cos().contiguous(), fr.sin().contiguous()


def fused_qkv(B, S, Hq, Hkv, dh, seed):
    """q / k / v as column views of one [B*S, (Hq + 2 Hkv) dh] buffer, as the decoder's fused QKV projection leaves them."""
    Dq, Dkv = Hq * dh, Hkv * dh
    buf = randn(B * S, Dq + 2 * Dkv, seed=seed).to(BF16)
    return (buf, buf[:, :Dq].view(B, S, Hq, dh), buf[:, Dq:Dq + Dkv].view(B, S, Hkv, dh), buf[:, Dq + Dkv:Dq + 2 * Dkv].view(B, S, Hkv, dh))


def padding_mask(S, pads):
    """key mask u8 [B, S] from (left, right) padding per sample; right = None: only key `left` is valid (a one-key sample)."""
    m = torch.zeros(len(pads), S, dtype=torch.uint8, device=dev())
    for i, (left, right) in enumerate(pads):
        if right is None:
            m[i, left] = 1
        else:
            m[i, left:S - right] = 1
    return m


def visible(B, Sq, Sk, causal, key_mask):
    """bool [B, 1, Sq, Sk]: query row i may attend key j."""
    vis = torch.ones(B, 1, Sq, Sk, dtype=torch.bool, device=dev())
    if causal:
        vis &= torch.ones(Sq, Sk, dtype=torch.bool, device=dev()).tril()
    if key_mask is not None:
        vis &= key_mask.bool()[:, None, None, :]
    return vis


def unrotate(g, cos, sin):
    """R^T g for HF rotate-half RoPE at position = token index: the gradient w.r.t. the un-rotated projection."""
    dh = g.shape[-1]
    c = torch.cat([cos, cos], -1).double()[None, :, None, :]
    s = torch.cat([sin, sin], -1).double()[None, :, None, :]
    return g * c + torch.cat([g[..., dh // 2:], -g[..., :dh // 2]], -1) * s


def reference(q, k, v, *, causal, scale, key_mask, dout=None, rope=None):
    """fp64 attention with explicit masking, GQA through repeat_interleave and autograd for the gradients.  A query row that sees no key
    has out = 0, lse = 0 and no gradient (the kernels' contract)."""
    B, Sq, Hq, dh = q.shape
    Sk, Hkv = k.shape[1], k.shape[2]
    qd, kd, vd = (t.detach().double().requires_grad_(dout is not None) for t in (q, k, v))
    kh = kd.transpose(1, 2).repeat_interleave(Hq // Hkv, dim=1)
    vh = vd.transpose(1, 2).repeat_interleave(Hq // Hkv, dim=1)
    s = (qd.transpose(1, 2) @ kh.transpose(-1, -2)) * scale
    s = s.masked_fill(~visible(B, Sq, Sk, causal, key_mask), float("-inf"))
    m = s.detach().amax(-1, keepdim=True)
    m = torch.where(torch.isfinite(m), m, torch.zeros_like(m))
    e = torch.exp(s - m)
    l = e.sum(-1, keepdim=True)
    out = ((e @ vh) / torch.where(l > 0, l, torch.ones_like(l))).transpose(1, 2)
    ld = l.detach()[..., 0]
    lse = torch.where(ld > 0, m[..., 0] + torch.log(torch.where(ld > 0, ld, torch.ones_like(ld))), torch.zeros_like(ld))
    grads = None
    if dout is not None:
        out.backward(dout.double())
        dq, dk, dv = qd.grad, kd.grad, vd.grad
        if rope is not None:
            dq, dk = unrotate(dq, *rope), unrotate(dk, *rope)
        grads = (dq, dk, dv)
    return out.detach(), lse, grads


def row_err(got, want, floor):
    """[B, S, H, dh] -> worst per-row relative error; rows are measured against at least `floor` x the largest row of their (sample, head)."""
    diff = (got.double() - want).abs().amax(-1)
    mag = want.abs().amax(-1)
    den = torch.maximum(mag, torch.maximum(mag.amax(dim=1, keepdim=True) * floor, mag.max() * TENSOR_FLOOR))
    return (diff / den).max().item()


def min_cos(got, want):
    """[B, S, H, dh] -> smallest cosine over the (sample, head) slices whose reference is not zero."""
    g, w = got.double().transpose(1, 2).flatten(2), want.transpose(1, 2).flatten(2)
    wn = w.norm(dim=-1)
    c = (g * w).sum(-1) / (g.norm(dim=-1) * wn).clamp_min(1e-300)
    return c[wn > 0].min().item()


def check_tensor(name, got, want, tol, zero_rows, floor=GRAD_FLOOR):
    """zero_rows bool [B, S, 1]: rows that must be exactly 0 (query rows that see no key; masked keys for dK / dV)."""
    assert torch.isfinite(got).all(), f"{name}: non-finite values"
    assert (got[zero_rows.expand(got.shape[:3])] == 0).all(), f"{name}: rows that see no key / masked keys are not exactly 0"
    err, cos = row_err(got, want, floor), min_cos(got, want)
    print(f"{name}: row err {err:.3e} (tol {tol:.1e}), min cos {cos:.6f}")
    assert err <= tol, (name, err)
    assert cos >= COS_MIN, (name, cos)


def check_lse(lse, want, no_key):
    assert (lse.transpose(1, 2)[no_key] == 0).all(), "lse of rows that see no key is not 0"
    excess = ((lse.double() - want).abs() - LSE_REL * want.abs()).max().item()
    print(f"lse: max |err| - {LSE_REL:.0e}|lse| = {excess:.3e} (tol {LSE_ABS:.1e})")
    assert excess <= LSE_ABS, excess


def run_and_check(q, k, v, *, causal, key_mask, dout_seed, backward=True, rope=True, out=None, grads_out=None, tol_grad=TOL_GRAD):
    """Forward (+ lse), then the backward with inverse RoPE where the shape allows it, all against the fp64 reference.
    Returns (out, lse, dq, dk, dv) of the kernels."""
    from slam_llm_b200 import ops
    B, Sq, Hq, dh = q.shape
    Sk = k.shape[1]
    scale = 1.0 / math.sqrt(dh)
    o, lse = ops.attn_fwd(q, k, v, causal=causal, scale=scale, key_mask=key_mask, out=out, need_lse=True)
    tables = rope_tables(Sq, dh) if (rope and Sq == Sk) else None
    dout = randn(B, Sq, Hq, dh, seed=dout_seed).to(BF16) if backward else None
    want_o, want_lse, want_g = reference(q, k, v, causal=causal, scale=scale, key_mask=key_mask, dout=dout, rope=tables)
    no_key = ~visible(B, Sq, Sk, causal, key_mask).any(-1)[:, 0]                # [B, Sq]
    masked_key = key_mask == 0 if key_mask is not None else torch.zeros(B, Sk, dtype=torch.bool, device=dev())
    check_tensor("out", o, want_o, TOL_OUT, no_key[..., None], OUT_FLOOR)
    check_lse(lse, want_lse, no_key)
    if not backward:
        return o, lse, None, None, None
    dq, dk, dv = ops.attn_bwd(q, k, v, o, lse, dout, causal=causal, scale=scale, key_mask=key_mask, rope=tables, **(grads_out or {}))
    for name, got, want, zero in zip(("dq", "dk", "dv"), (dq, dk, dv), want_g, (no_key, masked_key, masked_key)):
        check_tensor(name, got, want, tol_grad, zero[..., None])
    return o, lse, dq, dk, dv


# ------------------------------------------------------------------------------------------------- 1. large and rising logits
@pytest.mark.parametrize("B,S,Hq,Hkv,dh,causal,masked", [
    (2, 401, 8, 2, 128, True, True),      # decoder: tcgen05 forward and backward, GQA 4:1
    (2, 700, 4, 4, 64, False, False),     # encoder: tcgen05 forward
    (2, 60, 4, 2, 64, True, True),        # short: mma.sync forward and backward
])
def test_large_rising_logits(B, S, Hq, Hkv, dh, causal, masked):
    """q scaled by 7 (logits of ~7 sigma), plus a key-index ramp along head dimension 0 that raises the scores by ~8 (natural log) per
    128 keys, so the running maximum moves by more than 2^8 on every tile and the tcgen05 kernel's lazy TMEM rescale runs on every tile;
    plus one attention-sink key ~20 above everything else in a late tile."""
    _, q, k, v = fused_qkv(B, S, Hq, Hkv, dh, seed=101)
    ramp = torch.arange(S, device=dev(), dtype=F32) * (8.0 / 128.0) / (40.0 / math.sqrt(dh))   # scale * 40 * ramp = 8 per 128 keys
    sink = (3 * S) // 4
    qf, kf = q.float() * 7.0, k.float()
    qf[..., 0] += 40.0                                            # q . e0 = 40 +- 7: every query sees the rising ramp
    kf[..., 0] += ramp[None, :, None]
    kf[:, sink, :, 0] += 20.0 / (40.0 / math.sqrt(dh)) + float(ramp[-1] - ramp[sink])
    q.copy_(qf.to(BF16))
    k.copy_(kf.to(BF16))
    key_mask = padding_mask(S, [(7, 0)] + [(0, 5)] * (B - 1)) if masked else None
    if causal:
        # peaked rows (one key with P ~ 1): dS = P (dP - delta) is a difference of nearly equal terms and delta carries the 2^-9 rounding
        # of the bf16 output, so dQ / dK err up to 1.7e-2 of their (sample, head) here: held to the 3e-2 of the per-tensor check instead
        run_and_check(q, k, v, causal=True, key_mask=key_mask, dout_seed=102, tol_grad=3.0e-2)
    else:
        from slam_llm_b200 import ops
        run_and_check(q, k, v, causal=False, key_mask=key_mask, dout_seed=102, backward=False)
        # the encoder runs without lse: the unmasked tcgen05 kernel instance
        o, _ = ops.attn_fwd(q, k, v, causal=False, scale=1.0 / math.sqrt(dh))
        want, _, _ = reference(q, k, v, causal=False, scale=1.0 / math.sqrt(dh), key_mask=None)
        check_tensor("out (no lse)", o, want, TOL_OUT, torch.zeros(B, S, 1, dtype=torch.bool, device=dev()), OUT_FLOOR)


# ------------------------------------------------------------------------------------------------- 2. long padding, rows without keys
LONG_PADS = [(0, 0), (63, 0), (64, 0), (128, 0), (200, 0), (0, 130), (150, None)]


@pytest.mark.parametrize("Sq,Hq,Hkv,dh,causal", [
    (401, 8, 2, 128, True),       # tcgen05 forward + backward
    (401, 4, 2, 64, True),        # tcgen05 forward + mma.sync backward
    (401, 8, 2, 128, False),      # non-causal, Sq == Sk: tcgen05 forward + backward, plus a sample with every key masked
    (37, 4, 2, 64, False),        # non-causal, Sq != Sk: mma.sync forward + backward
])
def test_long_padding(Sq, Hq, Hkv, dh, causal):
    """Left padding of 0 / 63 / 64 / 128 / 200 keys, right padding of 130 and a one-key sample in one batch: whole 64-key (mma.sync) and
    128-key (tcgen05) tiles are masked.  Query rows that see no key (left-padded rows under the causal mask, every row of an all-masked
    sample) must give out = 0 and lse = 0 exactly, dQ = 0 exactly, and finite gradients everywhere."""
    Sk = 401
    pads = LONG_PADS + ([] if causal else [(Sk, 0)])
    B = len(pads)
    key_mask = padding_mask(Sk, pads)
    if Sq == Sk:
        _, q, k, v = fused_qkv(B, Sk, Hq, Hkv, dh, seed=201)
    else:
        q = randn(B, Sq, Hq, dh, seed=202).to(BF16)
        k, v = randn(B, Sk, Hkv, dh, seed=203).to(BF16), randn(B, Sk, Hkv, dh, seed=204).to(BF16)
    o, lse, dq, _, _ = run_and_check(q, k, v, causal=causal, key_mask=key_mask, dout_seed=205)
    no_key = ~visible(B, Sq, Sk, causal, key_mask).any(-1)[:, 0]       # [B, Sq]
    assert no_key.any()
    assert (o[no_key] == 0).all() and (lse.transpose(1, 2)[no_key] == 0).all() and (dq[no_key] == 0).all()


# ------------------------------------------------------------------------------------------------- 3. masked keys are invisible
@pytest.mark.parametrize("Sq,Sk,Hq,Hkv,dh,causal", [
    (300, 300, 8, 2, 128, True),  # tcgen05 forward + backward
    (300, 300, 4, 2, 64, True),   # tcgen05 forward + mma.sync backward
    (1, 300, 8, 2, 128, False),   # decode: mma.sync forward + backward
])
def test_masked_keys_invisible(Sq, Sk, Hq, Hkv, dh, causal):
    """K / V rows at masked positions replaced by +-3e4 (bf16-exact): out and lse bit-identical, dK / dV at masked keys exactly 0, the rest
    of the gradients within tolerance of the reference (dQ goes through fp32 atomics: not bit-reproducible)."""
    from slam_llm_b200 import ops
    pads = [(0, 0), (70, 0), (0, 140), (130, 20)]
    B = len(pads)
    key_mask = padding_mask(Sk, pads)
    if Sq == Sk:
        _, q, k, v = fused_qkv(B, Sk, Hq, Hkv, dh, seed=301)
    else:
        q = randn(B, Sq, Hq, dh, seed=302).to(BF16)
        k, v = randn(B, Sk, Hkv, dh, seed=303).to(BF16), randn(B, Sk, Hkv, dh, seed=304).to(BF16)
    scale = 1.0 / math.sqrt(dh)
    o0, lse0 = ops.attn_fwd(q, k, v, causal=causal, scale=scale, key_mask=key_mask, need_lse=True)
    o0, lse0 = o0.clone(), lse0.clone()
    big = torch.where(torch.arange(dh, device=dev()) % 2 == 0, 3.0e4, -3.0e4).to(BF16)
    masked = key_mask == 0
    k[masked] = big
    v[masked] = -big
    o, lse, _, dk, dv = run_and_check(q, k, v, causal=causal, key_mask=key_mask, dout_seed=305)
    assert torch.equal(o, o0) and torch.equal(lse, lse0)
    assert (dk[masked] == 0).all() and (dv[masked] == 0).all()


# ------------------------------------------------------------------------------------------------- 4. decode: Sq != Sk
@pytest.mark.parametrize("Hq,Hkv,dh", [(32, 8, 128), (14, 2, 64)])
@pytest.mark.parametrize("Sk", [1, 2, 63, 64, 65, 128, 129, 600])
def test_decode_step_shape(Sk, Hq, Hkv, dh):
    """One new token per sequence against a KV cache of Sk positions, as LlamaLoRAB200.decode_step passes it: q contiguous [n, 1, Hq, dh],
    K and V separate contiguous [n, Sk, Hkv, dh] buffers, non-causal, a per-row key mask (left padding differs per row; the last
    position, the new token, is always valid)."""
    n = 8
    pads = [(min(p, Sk - 1), 0) for p in (0, 1, 5, 63, 64, 100, 129, 599)]
    key_mask = padding_mask(Sk, pads)
    q = randn(n, 1, Hq, dh, seed=400 + Sk).to(BF16)
    k = randn(n, Sk, Hkv, dh, seed=401 + Sk, scale=2.0).to(BF16)
    v = randn(n, Sk, Hkv, dh, seed=402 + Sk).to(BF16)
    run_and_check(q, k, v, causal=False, key_mask=key_mask, dout_seed=403, backward=False)


@pytest.mark.parametrize("Hq,Hkv,dh", [(32, 8, 128), (14, 2, 64)])
def test_noncausal_sq_ne_sk(Hq, Hkv, dh):
    """General non-causal Sq = 5 against Sk = 300 keys with padding, forward and backward (mma.sync kernels)."""
    pads = [(0, 0), (100, 0), (0, 171)]
    q = randn(3, 5, Hq, dh, seed=410).to(BF16)
    k, v = randn(3, 300, Hkv, dh, seed=411).to(BF16), randn(3, 300, Hkv, dh, seed=412).to(BF16)
    run_and_check(q, k, v, causal=False, key_mask=padding_mask(300, pads), dout_seed=413)


# ------------------------------------------------------------------------------------------------- 5. GQA group size 7
@pytest.mark.parametrize("Hq,Hkv,dh", [(14, 2, 64), (28, 4, 128)])     # Qwen2-0.5B / Qwen2-7B attention
@pytest.mark.parametrize("S", [150, 401])
def test_gqa_group7(S, Hq, Hkv, dh):
    """A group size that is not a power of two: tcgen05 forward + mma.sync backward (dh 64), tcgen05 both ways (dh 128)."""
    _, q, k, v = fused_qkv(2, S, Hq, Hkv, dh, seed=500 + S)
    run_and_check(q, k, v, causal=True, key_mask=padding_mask(S, [(9, 0), (0, 13)]), dout_seed=501)


# ------------------------------------------------------------------------------------------------- 7. production gradient layout
@pytest.mark.parametrize("Hq,Hkv,dh", [(8, 2, 128), (8, 8, 128), (14, 2, 64)])
def test_fused_gradient_layout(Hq, Hkv, dh):
    """The training step's layout: q / k / v and dq / dk / dv are column views of fused [B*S, Dq + 2 Dkv (+ guard)] buffers and the forward
    output has a wider row stride too.  The gradient buffer is pre-filled with NaN: every gradient element is written, and the 64 guard
    columns (32 between dq and dk, 32 after dv) are never touched."""
    B, S = 2, 257
    Dq, Dkv = Hq * dh, Hkv * dh
    _, q, k, v = fused_qkv(B, S, Hq, Hkv, dh, seed=701)
    out_buf = torch.full((B * S, Dq + 64), float("nan"), device=dev(), dtype=BF16)
    g = torch.full((B * S, Dq + 2 * Dkv + 64), float("nan"), device=dev(), dtype=BF16)
    views = dict(dq=g[:, :Dq].view(B, S, Hq, dh), dk=g[:, Dq + 32:Dq + 32 + Dkv].view(B, S, Hkv, dh),
                 dv=g[:, Dq + 32 + Dkv:Dq + 32 + 2 * Dkv].view(B, S, Hkv, dh))
    _, _, dq, dk, dv = run_and_check(q, k, v, causal=True, key_mask=padding_mask(S, [(30, 0), (0, 40)]), dout_seed=702,
                                     out=out_buf[:, :Dq].view(B, S, Hq, dh), grads_out=views)
    assert dq.data_ptr() == views["dq"].data_ptr() and dk.data_ptr() == views["dk"].data_ptr() and dv.data_ptr() == views["dv"].data_ptr()
    assert torch.isnan(out_buf[:, Dq:]).all()
    assert torch.isnan(g[:, Dq:Dq + 32]).all() and torch.isnan(g[:, Dq + 32 + 2 * Dkv:]).all()
