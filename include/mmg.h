/*
 * mmg.h — C-ABI of libmmg.so: hand-written sm_100a kernels for the MaskGit.generate() hot path.
 *
 * This is the drop-in boundary (SURVEY.md section 8b, "lower face").  Every entry point is
 *     extern "C" int mmg_<op>(const mmg_<op>_args* a, void* cuda_stream);
 * with a POD argument block of raw DEVICE pointers + sizes.  Conventions:
 *   - returns 0 on success, a negative MMG_E* code otherwise; never throws, never allocates device memory,
 *     never synchronises the host; asynchronous on `cuda_stream` (a cudaStream_t) and CUDA-graph capturable;
 *   - no ownership transfer; the caller (PyTorch) owns all buffers;
 *   - mmg_last_error() returns a thread-local, human readable description of the last failure;
 *   - activations are row-major "token-major" matrices [rows, channels] (images: NHWC); `dtype` selects the
 *     operand type of a matrix product: MMG_BF16 -> tcgen05 tensor-core path (fp32 accumulate in TMEM),
 *     MMG_F32 -> fp32 CUDA-core path ("parity precision").  There is no CPU path in this library.
 *
 * Each function cites the reference code it replaces (paths relative to /root/reference/muse_maskgit_pytorch/).
 */
#ifndef MMG_H_
#define MMG_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MMG_VERSION 100

/* error codes */
#define MMG_OK            0
#define MMG_EINVAL       -1   /* bad argument / unsupported shape */
#define MMG_ECUDA        -2   /* CUDA runtime / driver error (see mmg_last_error) */
#define MMG_EUNSUPPORTED -3   /* device is not sm_100 */

/* operand dtypes */
#define MMG_F32  0
#define MMG_BF16 1

int         mmg_version(void);
const char* mmg_last_error(void);
/* Number of kernel launches issued through this library by the calling process (bench.py "gpu_launches"). */
int64_t     mmg_launch_count(void);
/* Number of bf16 matrix products / convolutions of this process that fell off the tcgen05 path onto the CUDA-core kernel because of their shape
 * or alignment (K or Cin % 64, N % 64, 16-byte rows, conv tile geometry).  MMG_VERBOSE=1 logs each one to stderr. */
int64_t     mmg_simt_fallback_count(void);
/* Number of launches of the CUDA-core matrix-product / attention kernels (any dtype) by this process.  precision="fp32" runs its products on the
 * tensor cores as 3-way bf16 splits (mmg_split3), so this stays 0 for a model whose shapes the TMA path takes. */
int64_t     mmg_simt_launch_count(void);
/* sizeof() of the argument block of entry point `name` ("mmg_linear", ...; "mmg_epilogue" for mmg_epilogue_args): lets a
 * foreign-language binding verify its struct mirror. Returns 0 for unknown names. */
int         mmg_sizeof(const char* name);

/* ------------------------------------------------------------------------------------------------
 * Matrix product with fused epilogue:  C[M,N] = A[M,K] * W[N,K]^T  (+ epilogue)
 * replaces: every nn.Linear on the path (muse_maskgit_pytorch.py:85,88,118,119,124,225,233) and, through
 * mmg_conv2d / mmg_conv_transpose2d below, every nn.Conv2d / nn.ConvTranspose2d (vqgan_vae.py:224-232,255-277).
 * ---------------------------------------------------------------------------------------------- */
enum mmg_epilogue {
  MMG_EPI_STORE      = 0, /* out[r, c] = acc (+bias[c]) (+leaky_relu 0.1 if act==1); out dtype = out_dtype          */
  MMG_EPI_RESIDUAL   = 1, /* out[r, c] = acc (+bias[c]) + resid[r, c]; out/resid dtype = out_dtype (may alias)      */
  MMG_EPI_GEGLU      = 2, /* W rows interleaved in blocks of 32: [x(32) | gate(32)]; out[r, c/2] = gate*gelu_erf(x) */
  MMG_EPI_GLU        = 3, /* same interleave, with bias: out = (a+ba) * sigmoid(g+bg)         (nn.GLU, vqgan_vae.py:256) */
  MMG_EPI_QKV        = 4, /* N = (nq+nk+nv)*64 head-columns: l2norm(q)*q_scale, l2norm(k)*k_scale, v -> per-head layouts */
  MMG_EPI_CONVT      = 5, /* conv-transpose parity scatter: out pixel (2y+py, 2x+px) = leaky(acc + bias)             */
  MMG_EPI_CONVT_RGB  = 6, /* CONVT followed by the fused final 1x1 conv (C -> channels<=4), fp32 NCHW output          */
  MMG_EPI_LNFOLD_RESIDUAL = 7, /* LayerNorm folded through the product: with W' = W*gamma, cvec[c] = sum_k W'[c,k] (passed as
                                  `bias`) and per-row (sum, sumsq) of the un-normalised A row in `row_stats`:
                                  out[r,c] = resid[r,c] + rstd_r * (acc - mean_r * cvec[c])   == resid + LN(a_r) W^T           */
  MMG_EPI_LFQ_IDS    = 8, /* LFQ lookup fused into the projection: W rows = [hi(bits) | mid(bits) | lo(bits)] (a 3-way bf16 split
                             of the fp32 project_in weight, 3*bits <= 64 = N), bias = project_in bias [bits], ln_width = bits:
                             ids[r] = sum_i ((hi+mid+lo)_i + bias_i > 0) << (bits-1-i), written as int64 to out[r]                */
  MMG_EPI_ARGMIN     = 9, /* nearest codebook row: W = codebook [K, D], bias = ||e_k||^2 [K]; out = uint64 best[M], initialised to
                             all-ones by the caller, updated with atomicMin( orderkey(||e||^2 - 2 x.e) << 32 | k ): lowest k on ties */
};

typedef struct {
  void*        out;        /* see enum; [M, ldo]                                                                 */
  int64_t      ldo;        /* leading dimension of out (elements)                                                */
  int32_t      out_dtype;  /* MMG_F32 / MMG_BF16                                                                 */
  int32_t      act;        /* 0 none, 1 leaky_relu(0.1)                                                          */
  const float* bias;       /* [N] or NULL (for GEGLU/GLU: interleaved like W rows)                               */
  const void*  resid;      /* RESIDUAL: [M, ldr] of out_dtype                                                    */
  int64_t      ldr;
  /* QKV: q -> q_out[(b*heads+h), t, 64]; k,v -> k_out/v_out[(b*heads+h), key_off + t, 64] with row r = b*tokens + t */
  void*        q_out; void* k_out; void* v_out;   /* dtype = out_dtype                                            */
  const float* q_scale; const float* k_scale;     /* [64]                                                         */
  const void*  null_k; const void* null_v;        /* optional [heads, 64] of out_dtype: written to key row 0 of every
                                                     (b, h) by the thread that owns token 0 (learned null key/value) */
  int32_t      heads, tokens, q_rows, kv_rows, key_off, nq_heads, nk_heads, nv_heads;
  /* CONVT(_RGB): input geometry of the GEMM rows (b, y, x) and the output parity                                  */
  int32_t      H, W, py, px;
  /* Fused LayerNorm of the OUTPUT row (RESIDUAL / LNFOLD_RESIDUAL with N == 2 tile widths, bf16 tensor-core path): besides
   * out = epilogue(acc) + resid the kernel also writes ln_out[r, :] = LN(out[r, :]) * gamma as bf16 for the next matrix product.
   * Rows >= ln_split first get out += ln_add[:] and use ln_gamma_b (null-CFG rows whose cross-attention is the constant
   * to_out(null_v)).  The two CTAs that own the halves of a row exchange (sum, sumsq) through distributed shared memory.  */
  void*        ln_out; int64_t ld_ln;
  const float* ln_gamma; const float* ln_gamma_b; const float* ln_add; int64_t ln_split;
  float*       row_stats;  /* [M, stats_slots, 2] fp32 (sum, sum of squares) partials.  GEGLU: the epilogue WRITES the statistics of each
                              64-column accumulator chunk (32 outputs, as rounded to out_dtype) to slot col / 64 (stats_slots >= N / 64;
                              every slot of every row is written exactly once, no atomics); LNFOLD_RESIDUAL: adds the stats_slots partials
                              of its row in ascending order (statistics over ln_width columns, eps 1e-5) — bitwise reproducible           */
  int32_t      ln_width; int32_t stats_slots;
  const float* rgb_w;      /* CONVT_RGB: [channels, N] fp32 1x1 weights, rgb_b [channels]                          */
  const float* rgb_b;
  int32_t      rgb_channels;
  int32_t      _pad;
} mmg_epilogue_args;

typedef struct {
  const void* a;           /* [M, lda] operand dtype                                                             */
  const void* w;           /* [N, ldw] operand dtype (nn.Linear weight layout, K contiguous)                     */
  int64_t M, N, K, lda, ldw;
  int32_t dtype;           /* MMG_BF16: tcgen05 path (K % 64 == 0, N % 64 == 0, 16B-aligned rows); MMG_F32: CUDA cores */
  int32_t epilogue;        /* enum mmg_epilogue                                                                   */
  mmg_epilogue_args epi;
} mmg_linear_args;
int mmg_linear(const mmg_linear_args* a, void* stream);

/* Convolutions as implicit GEMM over NHWC activations; weights pre-packed [Cout, taps*Cin] (tap-major, Cin
 * contiguous).  kind: 0 = 1x1; 1 = 3x3 stride 1 pad 1; 2 = 4x4 stride 2 pad 1; 3 = 5x5 stride 1 pad 2.
 * replaces: nn.Conv2d at vqgan_vae.py:224,231,232,255,258,261,271,274,277.                                        */
typedef struct {
  const void* x;           /* [B, H, W, Cin]                                                                     */
  const void* w;           /* [Cout, taps*Cin]                                                                   */
  int32_t B, H, W, Cin, Cout, kind;
  int32_t dtype, epilogue; /* STORE / RESIDUAL / GLU                                                             */
  mmg_epilogue_args epi;   /* rows of `out` are output pixels (b, y, x) in NHWC order                            */
} mmg_conv2d_args;
int mmg_conv2d(const mmg_conv2d_args* a, void* stream);

/* ConvTranspose2d(k=4, s=2, p=1) as 4 parity-class GEMMs (K = 4*Cin each).  w: [4 parities][Cout, 4*Cin].
 * replaces: nn.ConvTranspose2d + LeakyReLU at vqgan_vae.py:225 (and, with CONVT_RGB, the 1x1 at vqgan_vae.py:232). */
typedef struct {
  const void* x;           /* [B, H, W, Cin]                                                                     */
  const void* w;           /* [4, Cout, 4*Cin]                                                                   */
  int32_t B, H, W, Cin, Cout;
  int32_t dtype, epilogue; /* CONVT or CONVT_RGB                                                                 */
  mmg_epilogue_args epi;   /* out: [B, 2H, 2W, Cout] (CONVT) or fp32 [B, channels, 2H, 2W] (CONVT_RGB)           */
} mmg_conv_transpose2d_args;
int mmg_conv_transpose2d(const mmg_conv_transpose2d_args* a, void* stream);

/* First encoder conv: k x k (odd k <= 9, padding k / 2; the reference default is 5), Cin = channels (<= 4), fp32 NCHW image in, NHWC act
 * out.  replaces vqgan_vae.py:231.                                                                                  */
typedef struct {
  const float* img;        /* [B, C, H, W] fp32                                                                  */
  const float* w;          /* [Cout, C, k, k] fp32 (reference layout)                                            */
  const float* bias;       /* [Cout]                                                                             */
  void*        out;        /* [B, H, W, Cout] out_dtype                                                          */
  int32_t B, C, H, W, Cout, out_dtype;
  int32_t ksize, _pad;     /* k; 0 = 5                                                                           */
} mmg_conv_in_args;
int mmg_conv_in(const mmg_conv_in_args* a, void* stream);

/* GroupNorm(groups, eps 1e-5) over NHWC, in place, optional LeakyReLU(0.1).  replaces vqgan_vae.py:257,260,272-276. */
typedef struct {
  void*        x;          /* [B, HW, C] dtype, normalised in place                                              */
  const float* gamma; const float* beta;
  int32_t B, HW, C, groups, dtype, act;
} mmg_groupnorm_args;
int mmg_groupnorm(const mmg_groupnorm_args* a, void* stream);

/* ------------------------------------------------------------------------------------------------
 * LayerNorm (eps 1e-5, gamma only — beta is a zero buffer): muse_maskgit_pytorch.py:63-70.
 *   y[r, :] = LN(x[r, :width] (+ add[:]) ) * gamma, columns >= width are written as 0 up to ldy.
 *   If x_out != NULL the (x + add) sum is also written back (fp32) — used for the constant null-CFG cross-attn term.
 * ---------------------------------------------------------------------------------------------- */
typedef struct {
  const void*  x;  int32_t x_dtype;  int32_t y_dtype;
  void*        y;
  const float* gamma;      /* [width]                                                                            */
  const float* add;        /* [width] or NULL                                                                    */
  float*       x_out;      /* fp32 [rows, ldx] or NULL                                                           */
  float*       zero_stats; /* optional [rows, 2]: reset to 0 (kept for callers that accumulate their own row statistics; the GEGLU
                              epilogue writes per-chunk partials and needs no reset)                                          */
  int64_t      add_from;   /* `add` / `x_out` apply to rows >= add_from only (null-CFG branch rows of a 2-branch batch)   */
  int64_t rows, width, ldx, ldy;
} mmg_layernorm_args;
int mmg_layernorm(const mmg_layernorm_args* a, void* stream);

/* x[r, :] = token_emb[ids[r]] + pos_emb[r % n]  (fp32): muse_maskgit_pytorch.py:322-323; `copies` replicas of the
 * whole [rows, dim] block are written back to back (cond / null CFG branches share the embedding).               */
typedef struct {
  const int64_t* ids; const float* token_emb; const float* pos_emb;
  float* x; int64_t rows, n, dim; int32_t copies; int32_t use_pos;
} mmg_embed_args;
int mmg_embed(const mmg_embed_args* a, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Attention core: out[b, t, h*64:(h+1)*64] = softmax(scale * q.k^T + key_mask) v   with dh = 64.
 * q [BH, Tq, 64], k/v [BH, Tk_alloc, 64] already l2-normalised/scaled (epilogue MMG_EPI_QKV); key 0 is the null key.
 * replaces: Attend.forward / flash_attn (attend.py:66-140) + the head split/merge in Attention.forward
 * (muse_maskgit_pytorch.py:143-161).  key_mask: [B, Tk - 1] uint8, one byte per real key 1 .. Tk-1 (1 = attend; the null key is never
 * masked) or NULL; masked logits = -FLT_MAX.
 * Padding: rows [Tk, Tk_alloc) of each k / v head may be read (the tensor-core kernels load whole key blocks, so the last block reads into
 * the padding, or into the next head's rows) but never reach the output: they, like masked keys, get a weight of exactly 0.  They and the
 * masked keys' rows must hold finite values: 0 * inf is NaN, and the kernels do not guard against it.  Zero padding (what MMG_EPI_QKV
 * leaves) is fine.                                                                                                  */
typedef struct {
  const void* q; const void* k; const void* v; void* out;
  const uint8_t* key_mask;
  int32_t B, heads, Tq, Tk, Tk_alloc, dtype;
  int64_t ldo;             /* out row stride (elements) = heads*64 normally                                      */
  int32_t kv_batch_stride_zero;  /* 1: k/v are shared by all batch entries (per head only)                        */
  float   scale;
  float   logit_bound;     /* optional: a guaranteed upper bound on |q.k| (for l2-normalised q, k: max_i |q_scale_i k_scale_i|);
                              > 0 lets the tensor-core kernel run a single-pass softmax against that fixed maximum. 0 = unknown. */
  int32_t split3;          /* 1 (with dtype MMG_BF16): fp32 parity on the tensor cores.  q, k, v are mmg_split3 outputs of the fp32 [.., 64] tensors
                              (384 bf16 columns per row: q with side 0, k and v with side 1), out is fp32; exact two-pass softmax.      */
} mmg_attention_args;
int mmg_attention(const mmg_attention_args* a, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Sampler.  replaces muse_maskgit_pytorch.py:556-609 (the per-step tail of MaskGit.generate).
 * ---------------------------------------------------------------------------------------------- */
/* re-mask: select the num_masked highest scores per batch row (ties: lowest position first), write mask_id there,
 * set all scores to -1e5, and emit the ascending list of masked positions (muse_maskgit_pytorch.py:561-563).     */
typedef struct {
  int64_t* ids; float* scores; int32_t* masked_pos;   /* [B, n], [B, n], [B, num_masked]                          */
  int32_t B, n, num_masked; int64_t mask_id;
} mmg_remask_args;
int mmg_remask(const mmg_remask_args* a, void* stream);

/* Final LayerNorm + classifier-free-guidance combine on the masked rows only, in embedding space:
 *   e[j] = LN(x_null[r]) + (LN(x_cond[r]) - LN(x_null[r])) * cond_scale,  r = b*n + masked_pos[b, j]
 * (to_logits is linear and bias-free, so W e == null + (cond - null) * scale of muse_maskgit_pytorch.py:254).    */
typedef struct {
  const float* x_cond; const float* x_null;  /* [B*n, dim] fp32; x_null may be NULL (cond_scale == 1)             */
  const float* gamma; const int32_t* masked_pos;
  void* e; int32_t e_dtype;
  int32_t B, n, num_masked, dim; float cond_scale;
} mmg_final_embed_args;
int mmg_final_embed(const mmg_final_embed_args* a, void* stream);

/* top-k filter + gumbel-argmax + confidence score for R logits rows (muse_maskgit_pytorch.py:576-609, 403-418):
 *   keep the k largest logits of each row (ties at the threshold: lowest index first);
 *   pred = argmax_v( logit_v / max(T, 1e-10) - log(-log(u_v)) ),   u clamped at 1e-20 as the reference's log();
 *   score = 1 - softmax(logits)[pred];  ids[b, pos] = pred;  scores[b, pos] = score.
 * Noise: `u` != NULL -> injected uniforms, u[(b*n + pos) * V + v] (parity mode: the tensor the reference would
 * draw); else Philox4x32-10(seed, counter = (global row, v)) so results do not depend on the GPU count.          */
typedef struct {
  const float* logits;     /* [R, V] fp32, R = B*num_masked, row j of batch b at b*num_masked + j                  */
  const int32_t* masked_pos;
  int64_t* ids; float* scores;             /* [B, n]                                                              */
  const float* u;          /* [B, n, V] or NULL                                                                   */
  int32_t B, n, num_masked, V, k;
  float temperature;
  uint64_t seed; uint64_t step; int64_t row_offset;  /* global row = row_offset + b*n + pos                        */
  const uint64_t* seed_dev;  /* optional device word added to `seed` at run time (lets a captured CUDA graph be replayed
                                with a fresh seed)                                                                   */
  int64_t mask_id; int32_t only_masked;         /* only_masked != 0: ids[b, pos] is replaced only where it equals mask_id (the
                                `where(is_mask, pred_ids, ids)` of :582-588 when rows of already-decoded positions are scored
                                too, can_remask_prev_masked = True); scores are written for every listed row              */
  int32_t rng_mode;          /* u == NULL only.  0: the keying above.  1: the stream ATen's CUDA `zeros_like(t).uniform_(0, 1)` draws
                                for the reference's [B_global, n, V] noise tensor (muse_maskgit_pytorch.py:407) from a generator with
                                seed (seed + *seed_dev) and offset (aten_offset + *aten_offset_dev): element i = t + aten_stride*k is
                                word k&3 of Philox(counter = offset/4 + k/4, subsequence = t) * 2^-32 + 2^-33, 1 -> 0; aten_stride =
                                256 * min(SMs * maxThreadsPerSM/256, ceil(numel/256)); accurate logf / IEEE division as with `u`  */
  uint64_t aten_offset; const uint64_t* aten_offset_dev; uint32_t aten_stride, _pad;
  /* optional row indirection (the fallback leg of mmg_logits_fused): logits row j belongs to sampled row row_index[j] (the index into
     masked_pos), only the first min(*row_count_dev, row_index_cap) rows are processed; the grid is row_index_cap CTAs               */
  const int32_t* row_index; const int32_t* row_count_dev; int32_t row_index_cap, _pad2;
} mmg_logits_sample_args;
int mmg_logits_sample(const mmg_logits_sample_args* a, void* stream);

/* to_logits + the sampling tail of a decode step in one call, WITHOUT a [rows, V] logits buffer (muse_maskgit_pytorch.py:576-609 on the rows
 * listed in s.masked_pos; bf16 operands, tcgen05): a 4096-column sample GEMM gives every row a candidate threshold, the logits GEMM's epilogue
 * keeps online-softmax partials and emits only the candidates >= threshold (~12 % of the logits) as per-row lists, a finishing kernel runs the
 * exact-rank perturbed argmax of mmg_logits_sample on the lists.  Rows whose threshold missed are redone through materialised logits inside the
 * same call (<= 128 rows per call; beyond that status[1] is raised and the caller must repeat the step with mmg_linear + mmg_logits_sample).
 * Same results as mmg_linear + mmg_logits_sample up to the summation order of the softmax denominator.                                        */
typedef struct {
  const void* e;           /* [rows, K] bf16: mmg_final_embed output, rows = s.B * s.num_masked                                 */
  const void* w;           /* [V, K] bf16 to_logits weight                                                                        */
  int32_t K, _pad;
  int64_t rows_capacity;   /* the R_max the workspace was sized for (0: rows of this call)                                        */
  mmg_logits_sample_args s;/* sampler arguments as for mmg_logits_sample; s.logits / s.row_index are ignored                      */
  void* workspace; uint64_t workspace_bytes;   /* >= mmg_logits_fused_workspace_bytes(rows_capacity, V, K, k), 256-byte aligned   */
  int32_t* status;         /* device int32[2], zeroed by the caller: [0] += rows redone through the materialised fallback,
                              [1] = 1 when a step had more such rows than the fallback holds (results of that step are incomplete)  */
} mmg_logits_fused_args;
/* 0 when the shape is not supported by the fused path (V % 256, V < 1024, K % 64, k too large for the candidate lists) */
uint64_t mmg_logits_fused_workspace_bytes(int64_t rows_capacity, int32_t V, int32_t K, int32_t k);
int mmg_logits_fused(const mmg_logits_fused_args* a, void* stream);

/* token-critic scoring branch of MaskGit.generate (muse_maskgit_pytorch.py:590-600; TokenCritic :383-386, SelfCritic :352-361):
 *   s[r] = dot(LayerNorm(x_cond[r]) * gamma, w) + bias;   x_null != NULL: s = s_null + (s - s_null) * cond_scale  (CFG, :257)
 *   scores[r] = s + (u[r] - 0.5) * noise_mul       noise_mul = critic_noise_scale * steps_until_x0 / timesteps
 * x_* are the residual streams after the critic's last block (the final LayerNorm and the 1-wide head are applied here).
 * u == NULL: u = Philox4x32-10(counter = (0xFFFFFFFF, step, row_offset + r), key = seed + *seed_dev) >> 8 * 2^-24.            */
typedef struct {
  const float* x_cond; const float* x_null;   /* [rows, dim] fp32; x_null may be NULL (cond_scale == 1, SelfCritic)   */
  const float* gamma; const float* w;         /* [dim] final LayerNorm gain, [dim] head weight (to_logits / to_pred)  */
  float bias, cond_scale, noise_mul; int32_t dim;
  const float* u;                             /* [rows] injected uniforms or NULL                                     */
  float* scores;                              /* [rows] out                                                           */
  int64_t rows, row_offset; uint64_t seed; const uint64_t* seed_dev; int32_t step;
  int32_t rng_mode;                           /* 1: ATen's `uniform(scores.shape)` stream (:598), see mmg_logits_sample_args */
  uint64_t aten_offset; const uint64_t* aten_offset_dev; uint32_t aten_stride, _pad;
} mmg_critic_score_args;
int mmg_critic_score(const mmg_critic_score_args* a, void* stream);

/* ------------------------------------------------------------------------------------------------
 * VQ lookup.  replaces the quantizer calls at vqgan_vae.py:424 and 429-435.
 * ---------------------------------------------------------------------------------------------- */
/* LFQ: ids[t] = sum_i (x[t,:].w_in[i,:] + b_in[i] > 0) << (bits-1-i)  — the nearest-codebook L2 argmin over {+-1}^bits. */
typedef struct {
  const void* x; int32_t dtype;            /* [T, D] token-major fmap                                              */
  const float* w_in; const float* b_in;    /* [bits, D], [bits]; NULL -> identity (D == bits)                     */
  int64_t* ids; int64_t T; int32_t D, bits;
  const void* w_split;                     /* optional, bf16 tokens: [64, D] bf16, rows [hi(bits) | mid(bits) | lo(bits) | 0...] = the 3-way bf16
                                              split of w_in (hi + mid + lo == w_in in fp32; 3 * bits <= 64, D % 64 == 0): the projection then
                                              runs on the tcgen05 path (mmg_linear + MMG_EPI_LFQ_IDS), one TMA stream over the tokens      */
} mmg_vq_lfq_encode_args;
int mmg_vq_lfq_encode(const mmg_vq_lfq_encode_args* a, void* stream);

/* explicit codebook: ids[t] = argmin_k ||x_t - e_k||^2 (first index on ties); 64x64 tiles staged through shared memory with
 * coalesced loads, per-row packed (distance, code) atomicMin across code tiles.  (Large problems: mmg_linear + MMG_EPI_ARGMIN.) */
typedef struct {
  const float* x; const float* codebook;   /* [T, D], [K, D] fp32                                                  */
  int64_t* ids; int64_t T; int32_t K, D;
} mmg_vq_l2_argmin_args;
int mmg_vq_l2_argmin(const mmg_vq_l2_argmin_args* a, void* stream);

/* ids -> codes -> project_out: out[t, :] = sum_i (+-1)_i * w_out[:, i] + b_out  (LFQ.indices_to_codes)            */
typedef struct {
  const int64_t* ids; const float* w_out; const float* b_out;   /* w_out [D, bits]                                 */
  void* out; int32_t dtype; int64_t T; int32_t D, bits;
} mmg_vq_decode_codes_args;
int mmg_vq_decode_codes(const mmg_vq_decode_codes_args* a, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Composite entry points: the launch sequences of one FeedForward and of one whole decode step, for hosts that want one call
 * per step.  They only issue the entry points above on `stream` (no allocation, no host sync, CUDA-graph capturable).
 * ---------------------------------------------------------------------------------------------- */
/* FeedForward of a block on `rows` rows, in place on the fp32 residual stream (muse_maskgit_pytorch.py:72-89), bf16 operands:
 *   xn = LN(x [+ add on rows >= add_from, written back]) * ln_gamma;  h = gate * gelu_erf(xn W1^T);  x += LN(h) * gamma_inner W2^T
 * (the inner LayerNorm is folded through the second product: w2f = W2 * gamma_inner, cvec = rowsum(w2f), MMG_EPI_LNFOLD_RESIDUAL). */
typedef struct {
  float* x; int64_t rows; int32_t dim, F, Fp;     /* x [rows, dim]; F = inner width int(dim*mult*2/3), Fp = F padded to a multiple of 64 */
  const float* ln_gamma;                          /* [dim]                                                                  */
  const void* w1;                                 /* [2*Fp, dim] bf16, rows interleaved in blocks of 32: [x(32) | gate(32)] */
  const void* w2f; const float* cvec;             /* [dim, Fp] bf16, [dim]                                                  */
  const float* add; int64_t add_from;             /* optional [dim] constant (to_out(null_v) of an all-masked cross-attention) */
  void* xn; void* h; float* stats;                /* workspace: [rows, dim] bf16, [rows, Fp] bf16, [rows, Fp / 32, 2] fp32   */
} mmg_ff_geglu_args;
int mmg_ff_geglu(const mmg_ff_geglu_args* a, void* stream);

/* One step of MaskGit.generate (muse_maskgit_pytorch.py:556-609) for the default path (bf16, no token critic, no self-conditioning):
 * re-mask -> embed -> depth x [self-attention, cross-attention, FeedForward] over `branches` copies of the batch (1, or 2 = cond + null
 * CFG; the first `live_branches` attend to the context, the others take the constant to_out(null_v)) -> final LayerNorm + CFG combine
 * on the masked rows -> logits GEMM -> top-k / gumbel argmax / confidence.  ids / scores / masked_pos are updated in place. */
typedef struct {
  const float* ln_gamma; const void* w_qkv;       /* self: [3*heads*64, dim]; cross: [heads*64, dim] (q only)                */
  const void* w_out;                              /* [dim, heads*64]                                                         */
  const float* q_scale; const float* k_scale;     /* [64]; k_scale, null_k, null_v: self-attention only                      */
  const void* null_k; const void* null_v;         /* [heads, 64] bf16: l2norm(null_k)*k_scale, null_v                        */
  float logit_bound; int32_t _pad;                /* max_i |q_scale_i k_scale_i| (+ slack), see mmg_attention_args           */
} mmg_attn_weights;
typedef struct {
  mmg_attn_weights self_attn, cross_attn;
  const void* ctx_k; const void* ctx_v;           /* this layer's context K/V [live*b*heads, ctx_alloc, 64] bf16 (null key at row 0), computed
                                                     once per generate() with mmg_linear + MMG_EPI_QKV                       */
  const float* cross_null_out;                    /* [dim] to_out(null_v)                                                    */
  const float* ff_ln_gamma; const void* ff_w1; const void* ff_w2f; const float* ff_cvec;
} mmg_layer_weights;
typedef struct {
  int32_t depth, dim, heads, n, V, F, Fp, b, branches, live_branches;
  const mmg_layer_weights* layers;                /* HOST array [depth]                                                      */
  const float* tok_emb; const float* pos_emb; const float* final_gamma; const void* w_logits;   /* fp32, fp32, fp32, [V, dim] bf16 */
  const uint8_t* ctx_key_mask; int32_t ctx_keys, ctx_alloc;   /* [live*b, ctx_keys] (1 = attend); keys incl. the null key = ctx_keys + 1 */
  int64_t* ids; float* scores; int32_t* masked_pos; int64_t mask_id;     /* [b, n], [b, n], [b, n] */
  int32_t num_masked, k_keep, step; float temperature, cond_scale; int32_t _pad;
  const float* u; uint64_t seed; const uint64_t* seed_dev; int64_t row_offset;   /* noise: see mmg_logits_sample_args        */
  void* workspace; uint64_t workspace_bytes;      /* >= mmg_decode_step_workspace_bytes(...), 256-byte aligned, ZERO-INITIALISED once by
                                                     the caller (the padding rows of the self-attention K/V stay zero)        */
} mmg_decode_step_args;
uint64_t mmg_decode_step_workspace_bytes(int32_t b, int32_t branches, int32_t n, int32_t dim, int32_t heads, int32_t Fp, int32_t V, int32_t max_masked);
int mmg_decode_step(const mmg_decode_step_args* a, void* stream);

/* dtype conversion / layout helpers used by the host mirror */
typedef struct { const void* src; void* dst; int64_t n; int32_t src_dtype, dst_dtype; } mmg_cast_args;
int mmg_cast(const mmg_cast_args* a, void* stream);

/* fp32 on the tensor cores (precision="fp32"): dst[r, 6K] bf16 = the hi / mid / lo bf16 terms of src[r, K] (hi + mid + lo == src to 24 bits),
 * ordered per `side` (0: left operand [lo|hi|mid|mid|hi|hi], 1: right operand [hi|lo|mid|hi|mid|hi]) so that one bf16 product of the two
 * 6K-wide operands accumulates lo*hi + hi*lo + mid*mid + mid*hi + hi*mid + hi*hi in fp32 = the fp32 product to ~2^-24.  An NHWC activation
 * is split per pixel (rows = B*H*W, K = Cin -> 6*Cin channels), a packed conv weight per (output channel, tap).
 * replaces: the fp32 arithmetic of nn.Linear / nn.Conv2d when parity with the fp32 reference is asked for (no reference counterpart). */
typedef struct { const float* src; void* dst; int64_t rows, K, lds; int32_t side, _pad; } mmg_split3_args;
int mmg_split3(const mmg_split3_args* a, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MMG_H_ */
