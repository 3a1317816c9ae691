/* slam_b200.h — C ABI of libslam_b200.so: the B200 (sm_100a) kernels behind the SLAM-LLM
 * training-step hot path (SURVEY.md §8a rows a1–a9).
 *
 * The reference (X-LANCE/SLAM-LLM) has NO native boundary: its hot path is PyTorch eager calls
 * into whisper / transformers / peft.  Each entry point below therefore cites the reference
 * Python call site (path:line under /root/reference) whose arithmetic it replaces; the Python
 * host mirror (src/slam_llm/…, slam_llm_b200/…) binds them through ctypes (INTEGRATION.md).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in _host;
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream);
 *   - tensors are row-major, innermost dimension contiguous, leading dimension in ELEMENTS;
 *   - bf16 = __nv_bfloat16 storage, f32 = float, i64 = int64_t, u8 = unsigned char;
 *   - return value: 0 on success, non-zero cudaError_t (or negative slam error) on failure;
 *     slam_last_error() returns a human-readable string for the last failure on this thread;
 *   - no entry point allocates, frees or synchronises: workspaces are caller-provided.
 */
#ifndef SLAM_B200_H_
#define SLAM_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SLAM_B200_ABI_VERSION 6

int slam_abi_version(void);
const char* slam_last_error(void);
/* number of kernel launches issued through this library since process start (bench "gpu_launches") */
int64_t slam_launch_count(void);

/* ---------------------------------------------------------------------------------------------
 * GEMM core (tcgen05 + TMEM accumulators, TMA-fed, persistent, warp-specialised).
 *   out[M,N] = act( alpha * ( A[M,K1]·B[N,K1]^T  +  A2[M,K2]·B2[N,K2]^T ) + bias[N] ) + residual[M,N]
 * Both operands are K-major bf16.  The optional second K-segment (A2,B2) is accumulated into the
 * SAME TMEM tile as the base product before the epilogue: this is the fused LoRA path, with
 * A2 = x·A_lora^T (rank-padded to a multiple of 64) and B2 = (alpha/r)·B_lora.
 * Replaces: F.linear in whisper/transformers + peft lora.Linear.forward
 *   (models/slam_model.py:214-218,400; models/encoder.py:26-27; models/projector.py:20-26).
 * -------------------------------------------------------------------------------------------*/
typedef struct slam_gemm_args {
  const void* a;   int64_t lda;   /* bf16 [M,K1] */
  const void* b;   int64_t ldb;   /* bf16 [N,K1] */
  int32_t k1;
  int32_t k2;                     /* 0 = no second segment */
  const void* a2;  int64_t lda2;  /* bf16 [M,K2] */
  const void* b2;  int64_t ldb2;  /* bf16 [N,K2] */
  void* out;       int64_t ldo;   /* bf16 or f32 [M,N] */
  int32_t out_f32;                /* 0: bf16 out, 1: f32 out */
  int32_t act;                    /* 0 none, 1 GELU(erf), 2 ReLU, 3 SwiGLU forward, 4 SwiGLU backward (see `aux`) */
  const float* bias;              /* f32 [N] or NULL */
  const void* residual; int64_t ldr; /* bf16 [M,N] or NULL; added after activation */
  float alpha;
  int32_t m, n;
  int32_t block_n;                /* tile override: 0 = auto; 64/128/192/256 = BLOCK_N with 128-row tiles;
                                     BLOCK_M*1000+BLOCK_N (e.g. 256256) = explicit 256-row tile;
                                     2000000+BLOCK_N (256/224/192/160/128) = CTA-pair kernel (cta_group::2: 256 x BLOCK_N per SM pair);
                                     3000064 = thin-product kernel (N <= 64: a cluster of 8 CTAs per 128-row tile splits K and reduces the
                                     partial tiles through distributed shared memory in a fixed order; what auto picks for such products) */
  int32_t split_k;                /* <= 1: off.  > 1: K is cut into that many slices processed by different CTAs and merged with
                                     fp32 atomics into `out`, which must be f32 and ZERO-INITIALISED by the caller; no bias /
                                     activation / residual (thin LoRA products, lm_head dgrad: few output tiles, long K) */
  void* workspace;                /* NULL, or slam_gemm_workspace_bytes() bytes of device memory, ZEROED ONCE by the caller and then
                                     owned by the library between calls on one stream (it leaves the flag area zeroed).  With a
                                     workspace the GEMM may "split the tail": the tiles of the last, partial wave are cut into
                                     k-slices run by otherwise idle SMs; the fp32 partial accumulators are exchanged through the
                                     workspace and added in a fixed order (deterministic), and the full epilogue (bias /
                                     activation / residual, bf16 or f32 out) still applies */
  int64_t workspace_bytes;
  int32_t tail_split;             /* 0 = automatic (when a workspace is given), -1 = never, n > 1 = at most n k-slices per tile */
  int32_t transpose_out;          /* 0: out[M,N] as above.  1 ("swap-AB"): `out` and `residual` are the TRANSPOSED matrices, bf16 [N,M] with row
                                     strides ldo / ldr: out[n][m] = sum_k A[m,k] B[n,k] (+ A2 B2) + residual[n][m].  The caller passes the WEIGHT
                                     as A (rows a multiple of 256: no padding in a CTA-pair tile) and the activations as B, so the token
                                     dimension becomes the flexible-width N of the tile and the result still lands as [tokens, features].
                                     Needs bf16 out, no bias, no split_k; act 0, or act 4 (SwiGLU backward, CTA-pair tiles): then A = W_down^T [F, d],
                                     B = dY [tokens, d], aux = gu [tokens, 2F], out = d(gu) [tokens, 2F] - 9 x 192 token columns instead of
                                     7 x 256 token rows: 12.5 % fewer tile-rounds at 1604 tokens */
  void* aux; int64_t ld_aux;      /* fused SwiGLU (HF LlamaMLP: down_proj(act_fn(gate_proj(x)) * up_proj(x)), modeling_llama.py), with the
                                     gate/up pair stored "blocked-64": feature 64 b + i has its gate in column 128 b + i and its up in
                                     column 128 b + 64 + i of a [M, 2F] matrix (weights pre-permuted by the caller to match).
                                     act 3: out = gu [M, N = 2F] as usual, and aux (bf16 [M, F], written) = silu(gate) * up computed from
                                            the bf16-rounded gu - identical to slam_swiglu_fwd on `out`;
                                     act 4: the product is dh [M, N = F] (never stored); aux (bf16 [M, 2F], read) = gu, and
                                            out (bf16 [M, 2F]) = d(gu) - identical to slam_swiglu_bwd(gu, bf16(dh)).
                                     Both need bf16 out, no bias / residual / split_k; act 3 needs tiles of 128 or 256 columns */
  int32_t static_operands;        /* bit 0: A, bit 1: B is CONSTANT for the lifetime of the stream's in-flight work (frozen weights - the
                                     reference's frozen encoder / LLM, models/slam_model.py:104-160): not written by any kernel that can still be
                                     running when this one starts.  The CTA-pair kernels then request the first ring of that operand's tiles
                                     BEFORE griddepcontrol.wait, i.e. under the tail of the preceding kernel (programmatic dependent launch), so
                                     the HBM latency of the first weight tiles is not paid after it (tools/gemm_trace.py: 2.6-3.3 us per launch).
                                     0 = nothing is assumed */
  int32_t reserved0;
} slam_gemm_args;
int slam_gemm_bf16(const slam_gemm_args* args, void* stream);
/* bytes of `workspace` the tail split needs on the current device (SM count x one 128 x 256 fp32 tile + flags) */
int64_t slam_gemm_workspace_bytes(void);

/* C[P,Q] (f32) = scale * sum_m A[m,P] * B[m,Q]   (thin weight-gradient product: P <= 64)
 * Used for LoRA dA / dB (peft lora.Linear backward) and bias gradients.  accumulate = 0: C is OVERWRITTEN;
 * accumulate != 0: the product is ADDED to C (the step zeroes its flat gradient buffer once instead of per product). */
int slam_wgrad_thin(const void* a_bf16, int64_t lda, int32_t p, const void* b_bf16, int64_t ldb,
                    int32_t q, int32_t m, float scale, float* c, int64_t ldc, int32_t accumulate, void* stream);

/* ---------------------------------------------------------------------------------------------
 * a1  log-mel front end.  whisper.pad_or_trim + whisper.log_mel_spectrogram(...).permute(1,0)
 *     as called at datasets/speech_dataset.py:101-103.
 *   wav      f32 [B, n_samples]  (padded/trimmed; n_frames = n_samples/160)
 *   lengths  i32 [B] real sample counts or NULL (= all n_samples).  With lengths, utterance b is transformed as if it had
 *            lengths[b] samples (reflect padding at ITS end, max over ITS frames) and its mel frames >= lengths[b]/160 are
 *            zero — the reference pads the mel, not the audio, in the dynamic-frame collator (speech_dataset_large.py:196-199)
 *   filters_t f32 [201, n_mels]  (slaney mel filterbank, TRANSPOSED so mel is the contiguous axis)
 *   out      f32 [B, n_frames, n_mels]
 *   scratch  f32 [B]  per-utterance running max (written by the kernel)
 * -------------------------------------------------------------------------------------------*/
int slam_logmel(const float* wav, int32_t batch, int32_t n_samples, const int32_t* lengths,
                const float* filters_t, int32_t n_mels, float* out, float* scratch_max, void* stream);

/* a2  Whisper conv stem helpers (models/encoder.py:18-24).  Time-major activations.
 *   im2col for Conv1d(k=3, pad=1, stride s): x[B,T,C] (f32 or bf16) -> col bf16 [B*T_out, ldk]
 *   with col[b,t,(kk*C + c)] = x[b, s*t + kk - 1, c] (zero outside); columns >= 3C zero-filled. */
int slam_conv_im2col(const void* x, int32_t x_is_f32, int32_t batch, int32_t t_in, int32_t c,
                     int32_t stride, void* col_bf16, int64_t ldk, void* stream);
/* y[b,t,:] = x[b,t,:] + pos[t,:]  (bf16 x, f32 pos) — models/encoder.py:24 */
int slam_add_pos(void* x_bf16, const float* pos, int32_t batch, int32_t t, int32_t d, void* stream);

/* LayerNorm over last dim (fp32 statistics), whisper LayerNorm / ln_post (models/encoder.py:26-29). */
int slam_layernorm(const void* x_bf16, const float* w, const float* b, void* y_bf16, int32_t rows,
                   int32_t d, float eps, void* stream);

/* Multi-head attention forward (flash-style, online softmax, bf16 in / fp32 accumulate).
 *   q [B,Sq,Hq,dh], k/v [B,Sk,Hkv,dh] given as base pointers + row strides (elements) so that the
 *   fused QKV buffer can be used in place.  causal: 0/1.  key_mask u8 [B,Sk] (1 = attend) or NULL.
 *   lse f32 [B,Hq,Sq] (log-sum-exp, natural log) or NULL.  out bf16 [B,Sq,Hq,dh] with row stride ldo.
 * Replaces whisper MultiHeadAttention.qkv_attention and HF LlamaAttention (eager softmax).
 * Kernels: tcgen05 / TMEM flash attention for dh = 64 / 128 with Sq == Sk >= 64 (forward) and dh = 128 (backward);
 * mma.sync flash kernels for every other shape - same arguments, same results within bf16 rounding.
 * Masking contract (both kernel families): a query row that sees no key (every key masked, or left padding under the causal mask)
 * gets out = 0 and lse = 0 exactly, and dQ = 0 exactly in the backward; a masked key gets dK = dV = 0 exactly, and the values
 * stored at masked K / V positions never reach out or lse (any finite values give bit-identical results). */
typedef struct slam_attn_args {
  const void* q; int64_t ldq;   /* row stride between consecutive tokens, elements */
  const void* k; int64_t ldk;
  const void* v; int64_t ldv;
  void* out;     int64_t ldo;
  float* lse;
  const uint8_t* key_mask;
  int32_t batch, sq, sk, hq, hkv, dh;
  int32_t causal;
  float scale;
  /* backward only */
  const void* dout; int64_t lddo;
  void* dq; int64_t lddq;
  void* dk; int64_t lddk;
  void* dv; int64_t lddv;
  float* delta;                  /* f32 [B,Hq,Sq] scratch */
  float* dq_accum;               /* f32 scratch [B,Sq,Hq,dh]: dQ partial sums (zeroed by the call) */
  void* dkv_part;                /* optional bf16 scratch [2,B,Sk,Hq,dh] (GQA only): per-Q-head dK/dV partials, summed over each
                                    KV group by a follow-up kernel -> Hq/Hkv times more CTAs; NULL = loop over the group in one CTA */
  const float* rope_cos;         /* optional f32 [>= max(sq, sk), dh/2] (both or neither): q and k were rotated by HF apply_rotary_pos_emb with */
  const float* rope_sin;         /* position = token index; the backward's finishing kernel then returns dQ / dK w.r.t. the UN-rotated q / k
                                    (inverse rotation fused with the GQA group sum and the fp32 -> bf16 conversion of dQ) */
} slam_attn_args;
int slam_attn_fwd(const slam_attn_args* a, void* stream);
int slam_attn_bwd(const slam_attn_args* a, void* stream);

/* a4  embedding gather + modality merge (models/slam_model.py:370-392).
 *   ids i64 [B,S] (-1 treated as 0), modality_mask u8 [B,S], audio bf16 [B,Ta,D],
 *   embed bf16 [V,D] -> x bf16 [B,S,D].  Semantics follow the reference loop exactly:
 *   start = argmax(mask), len = min(sum(mask), Ta); rows start..start+len-1 take audio rows;
 *   every other row r takes embed[ids[r]] * (mask[r] ? 0 : 1). */
int slam_embed_merge(const int64_t* ids, const uint8_t* modality_mask, const void* audio_bf16,
                     int32_t ta, const void* embed_bf16, void* x_bf16, int32_t batch, int32_t s,
                     int32_t d, void* stream);
/* backward of the merge wrt the audio rows: daudio[b,j,:] = dx[b,start+j,:] for j < len, else 0 */
int slam_embed_merge_bwd(const uint8_t* modality_mask, const void* dx_bf16, void* daudio_bf16,
                         int32_t ta, int32_t batch, int32_t s, int32_t d, void* stream);

/* full fine-tune (train_config.freeze_llm=false, models/slam_model.py:205-208 not taken; examples/s2s): gradients of the decoder's own
 * parameters that are not GEMM products.
 *   slam_rmsnorm_wgrad: dw[c] += sum_r dy[r,c] * x[r,c] * rstd[r]   (LlamaRMSNorm weight; dw f32 [d], ACCUMULATED: zero it first)
 *   slam_embed_grad:    dE[max(ids[r],0)] += dx[r] for rows with modality_mask[r] == 0  (embedding rows used by the merge, slam_model.py:392;
 *                       dE f32 [vocab, d], accumulated with atomics; rows = B*S) */
int slam_rmsnorm_wgrad(const void* dy_bf16, const void* x_bf16, const float* rstd, int32_t rows, int32_t d, float* dw, void* stream);
int slam_embed_grad(const int64_t* ids, const uint8_t* modality_mask, const void* dx_bf16, float* dE, int32_t rows, int32_t d,
                    int32_t vocab, void* stream);

/* a5  Llama decoder element-wise kernels (HF LlamaRMSNorm / apply_rotary_pos_emb / LlamaMLP). */
int slam_rmsnorm_fwd(const void* x_bf16, const void* w_bf16, void* y_bf16, float* rstd, int32_t rows,
                     int32_t d, float eps, void* stream);
/* dx = rmsnorm_bwd(dy; x, w, rstd) (+ dres if non-NULL): fuses the residual-stream gradient add */
int slam_rmsnorm_bwd(const void* dy_bf16, const void* x_bf16, const void* w_bf16, const float* rstd,
                     const void* dres_bf16, void* dx_bf16, int32_t rows, int32_t d, void* stream);
/* in-place rotate-half RoPE on heads laid out [rows, n_heads, dh] with row stride ld; position =
 * row % seq_len; cos/sin are f32 [seq_len, dh/2] tables (host builds them exactly like
 * LlamaRotaryEmbedding); inverse != 0 applies the transpose rotation (backward). */
int slam_rope(void* x_bf16, int64_t ld, int32_t rows, int32_t seq_len, int32_t n_heads, int32_t dh,
              const float* cos_table, const float* sin_table, int32_t inverse, void* stream);
/* h = silu(g) * u with gu bf16 [rows, 2F]; block = 0: gu = [g | u] (HF order of the concatenated gate/up weight);
 * block = 64: "blocked-64" order (see slam_gemm_args.aux), used when the fused GEMM epilogues are not */
int slam_swiglu_fwd(const void* gu_bf16, void* h_bf16, int32_t rows, int32_t f, int32_t block, void* stream);
int slam_swiglu_bwd(const void* gu_bf16, const void* dh_bf16, void* dgu_bf16, int32_t rows, int32_t f, int32_t block,
                    void* stream);

/* a6  LoRA-branch dropout (peft lora.Linear.forward: lora_B(lora_A(dropout(x))) — train_config.peft_config.lora_dropout).
 *   y = x * keep / (1-p) with keep(i) = hash(seed, i) >= p; the backward regenerates the same mask from (seed, i):
 *   out = base + lora * keep / (1-p)   (dX = dY W  +  mask o ((dY sB) A)).  n % 8 == 0; bf16. */
int slam_dropout(const void* x_bf16, void* y_bf16, int64_t n, float p, uint64_t seed, void* stream);
int slam_dropout_bwd_add(const void* base_bf16, const void* lora_bf16, void* out_bf16, int64_t n, float p, uint64_t seed,
                         void* stream);

/* a7  token cross-entropy + accuracy on fp32 logits rows (HF ForCausalLMLoss + utils/metric.py:3-20).
 *   logits f32 [R,V] (rows already shifted/selected by the host), targets i64 [R] (-100 = ignore).
 *   Outputs: loss_sum f32[1], n_valid i32 [1], n_correct i32 [1] (atomically accumulated: caller
 *   zeroes), and dlogits bf16 [R,V] = (softmax - onehot) * grad_scale[0] for valid rows, else 0.
 *   grad_scale is read from device memory so the 1/n_valid factor needs no host sync. */
int slam_cross_entropy(const float* logits, int64_t ldl, const int64_t* targets, int32_t rows,
                       int32_t vocab, float* loss_sum, int32_t* n_valid, int32_t* n_correct,
                       void* dlogits_bf16, int64_t lddl, const float* grad_scale, void* stream);

/* a8  AdamW on one flat f32 parameter buffer (torch.optim.AdamW, pipeline/finetune.py:247-251).
 *   step_host is the 1-based optimizer step; grad_div divides the gradient first (DDP mean). */
int slam_adamw(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, float lr,
               float beta1, float beta2, float eps, float weight_decay, int32_t step_host, float grad_div,
               void* stream);

/* utility kernels */
int slam_cast_f32_to_bf16(const float* x, void* y_bf16, int64_t n, float scale, void* stream);
int slam_cast_bf16_to_f32(const void* x_bf16, float* y, int64_t n, void* stream);
/* y[C,R] = x[R,C]^T (bf16) */
int slam_transpose_bf16(const void* x, int64_t ldx, void* y, int64_t ldy, int32_t rows, int32_t cols,
                        void* stream);
/* dst[b][j][i] = src[b][i][j] (f32): Conv1d weight-gradient layout [co,(k,c)] -> [co,c,k] of the cov1d projector */
int slam_transpose_f32_batched(const float* src, float* dst, int32_t batch, int32_t rows, int32_t cols, void* stream);
/* y[i,:] = x[idx[i],:]  /  y[idx[i],:] = x[i,:] (rows of d bf16; idx i32) */
int slam_gather_rows(const void* x_bf16, const int32_t* idx, void* y_bf16, int32_t n_idx, int32_t d,
                     void* stream);
int slam_scatter_rows(const void* x_bf16, const int32_t* idx, void* y_bf16, int32_t n_idx, int32_t d,
                      void* stream);
/* relu backward: dx = dy * (y > 0) ; bf16 */
int slam_relu_bwd(const void* dy_bf16, const void* y_bf16, void* dx_bf16, int64_t n, void* stream);
/* column sums: out[c] = sum_r x[r,c] (bf16 in, f32 out) — bias gradients */
int slam_colsum(const void* x_bf16, int64_t ldx, int32_t rows, int32_t cols, float* out, void* stream);
/* batched strided cast with optional transpose (packs LoRA adapters into rank-padded GEMM operands):
 *   dst[b][i][j] = scale*src[b][i][j]   (transpose == 0)    dst[b][j][i] = scale*src[b][i][j]  (transpose != 0) */
int slam_pack2d(const float* src, int64_t src_batch_stride, int64_t src_ld, void* dst_bf16,
                int64_t dst_batch_stride, int64_t dst_ld, int32_t batch, int32_t rows, int32_t cols,
                float scale, int32_t transpose, void* stream);
/* y = a + b (bf16) */
int slam_add_bf16(const void* a, const void* b, void* y, int64_t n, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SLAM_B200_H_ */
