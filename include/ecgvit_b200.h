/*
 * ecgvit_b200.h -- C ABI of the B200-native ECG-ViT training-step kernels.
 *
 * The reference (StefanHeng/ECG-Representation-Learning) has NO plugin / operator / FFI layer
 * (SURVEY.md 8b): its seam is the Python nn.Module API of `EcgVit`
 * (ecg_transformer/models/ecg_vit.py:95-149) and the step of `MyTrainer.train`
 * (ecg_transformer/models/train.py:268-283).  Each entry point below therefore cites the reference
 * (or un-vendored third-party `vit-pytorch==0.33.2`, requirements.txt:174) op sequence it replaces.
 *
 * Conventions
 *   - plain pointers and sizes; every pointer is a DEVICE pointer unless stated otherwise;
 *   - `dtype` selects the activation/operand type: ECGVIT_F32 (parity mode, FFMA contractions) or
 *     ECGVIT_BF16 (performance mode, tcgen05 contractions, fp32 accumulation and statistics);
 *   - parameters, optimizer state and gradients are always fp32;
 *   - the caller owns all memory; nothing is allocated, freed or retained past the call;
 *   - all work is stream-ordered on `stream` (a cudaStream_t cast to void*), no host sync, graph-capturable;
 *   - return value: 0 = ok, negative = invalid argument (see ecgvit_last_error), positive = cudaError_t.
 */
#ifndef ECGVIT_B200_H
#define ECGVIT_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ECGVIT_ABI_VERSION 7

/* ECGVIT_BF16_RES32: bf16 mode with an fp32 RESIDUAL STREAM (the running sum x / y of the blocks, which deep models such
 * as 'large' need to stay within 1e-2 of the fp32 reference).  Accepted by the entry points that touch the stream, which
 * then take that one operand as fp32: ecgvit_embed_assemble (tok), ecgvit_layernorm_fwd (x), ecgvit_layernorm_bwd (x),
 * ecgvit_head_fwd / ecgvit_head_bwd (tok); everything else they read or write stays bf16.  The Linear + residual GEMMs
 * use ECGVIT_EPI_BIAS_RES_F32. */
enum { ECGVIT_F32 = 0, ECGVIT_BF16 = 1, ECGVIT_BF16_RES32 = 2 };

/* GEMM epilogues */
enum {
    ECGVIT_EPI_STORE = 0,      /* out = acc (+ bias)                                              */
    ECGVIT_EPI_BIAS_RES = 1,   /* out = acc + bias + aux          (Linear + residual add)         */
    ECGVIT_EPI_BIAS_GELU = 2,  /* out = acc + bias ; out2 = gelu_erf(out)                         */
    ECGVIT_EPI_DGELU = 3,      /* out = acc * gelu_erf'(aux)                                      */
    ECGVIT_EPI_ATOMIC_F32 = 4, /* out(fp32) += acc                (weight gradients, split-K)     */
    ECGVIT_EPI_BIAS_RES_F32 = 5, /* out(fp32) = acc + bias + aux(fp32)  (bf16 GEMM, fp32 residual stream) */
    /* out = acc + bias - aux  (the residual of a prediction against the target `aux`, same dtype / ld as out) and
     * out2 = fp32 [ceil(N / 64), M] row partials of its square: out2[g * M + m] = sum over the columns
     * 64g .. min(64g + 64, N) - 1 of (acc + bias - aux)^2, taken in fp32 before out is rounded to dtype.  Plain stores,
     * no atomics, so the partials (and a loss folded from them in a fixed order) are bit-identical from run to run.
     * K-major A and B only; no dropout. */
    ECGVIT_EPI_BIAS_SUB_ROWSQ = 6
};

enum { ECGVIT_REDUCTION_MEAN = 0, ECGVIT_REDUCTION_SUM = 1, ECGVIT_REDUCTION_NONE = 2 };

int ecgvit_abi_version(void);
/* thread-local message for the last non-zero return of any entry point */
const char *ecgvit_last_error(void);
/* 1 when the current device is sm_100 (B200) */
int ecgvit_device_ok(void);

/* ---- patch embedding: replaces einops Rearrange 'b c (h p1) (w p2) -> b (h w) (p1 p2 c)' of
 *      vit_pytorch.ViT.to_patch_embedding[0] (call site ecg_vit.py:141).
 *      a[(b*n_patch + w), t*C + c] = x[b, c, w*P + t]   (bit-exact gather; cast to dtype)
 *      x is fp32 [B, C, x_ld] (x_ld >= n_patch*P elements per lead). */
int ecgvit_patchify(const float *x, void *a, int B, int C, int64_t x_ld, int n_patch, int P, int dtype,
                    void *stream);

/* ---- the same gather with the reference's per-record input pipeline fused in front (SURVEY 8f rank 1):
 *      preprocess/transform.py:18-35 Normalize ((x - mean[c]) / std[c], fp32 IEEE, bit-identical to numpy),
 *      :140-154 TimeEndPad (zeros from sample L_valid on, up to n_patch * P) and :175-185 TimeOut (zeros on
 *      [spans[2b], spans[2b] + spans[2b+1]) of every lead of record b), in the order EcgDataset.__getitem__ /
 *      ptb_dataset.py:132-149 apply them.  x [B, C, x_ld] raw fp32 records with L_valid <= x_ld samples per lead;
 *      mean / std device fp32[C] or both NULL; spans device int32[B, 2] or NULL. */
int ecgvit_patchify_transform(const float *x, const float *mean, const float *stdev, const int *spans, void *a,
                              int B, int C, int64_t x_ld, int L_valid, int n_patch, int P, int dtype,
                              void *stream);

/* ---- per-lead tokens (BASELINE.json configs[3]; the oracle is vit_pytorch's ViT(image_size=(C, L),
 *      patch_size=(1, P), channels=1) on [B, 1, C, L]): a[((b*C + c)*n_w + w), t] = x[b, c, w*P + t] for t < P and
 *      0 for P <= t < Kp (Kp = P rounded up to 8: the embedding GEMM reads 16-byte aligned rows).  mean / std / spans
 *      as in ecgvit_patchify_transform (all optional). */
int ecgvit_patchify_leads(const float *x, const float *mean, const float *stdev, const int *spans, void *a, int B,
                          int C, int64_t x_ld, int L_valid, int n_w, int P, int Kp, int dtype, void *stream);
/* helpers of that mode: zero-padded copy of a [rows, cols] matrix to [rows, cols_padded] (the embedding weight),
 * and dst[rows, cols] += src[rows, 0:cols] of a padded fp32 matrix (its gradient) */
int ecgvit_pad_cols(const void *src, void *dst, int64_t rows, int cols, int cols_padded, int dtype, void *stream);
int ecgvit_unpad_add_f32(const float *src, float *dst, int64_t rows, int cols, int cols_padded, void *stream);

/* ---- CLS concat + positional add: replaces torch.cat(cls, x); x += pos_embedding[:, :n+1]
 *      tok[b,0,:] = cls + pos[0];  tok[b,1+w,:] = e[b*n_patch+w,:] + pos[1+w]  (e already holds the bias) */
int ecgvit_embed_assemble(const void *e, const float *cls, const float *pos, void *tok, int B, int n_patch,
                          int d, float dropout_p, int dropout_stream, const uint32_t *dropout_seed, int dtype,
                          void *stream);
/* backward of the above (g = dropout mask applied to dtok): de = g[:,1:,:]; dpos += sum_b g; dcls += sum_b g[:,0];
 * dbias += sum_{b,w} g[:,1:] */
int ecgvit_embed_assemble_bwd(const void *dtok, void *de, float *dcls, float *dpos, float *dbias, int B,
                              int n_patch, int d, float dropout_p, int dropout_stream,
                              const uint32_t *dropout_seed, int dtype, void *stream);

/* ---- masked-patch pre-training (SimMIM-style: masked patches keep their place in the sequence).
 *      Added in ABI version 7 without changing any earlier entry point, so the version number stays 7.
 *
 *      Mask draw: patch w of record b is masked iff the rank of its key hash(seed, site, b*n_patch + w) (the 32-bit
 *      counter hash of the dropout masks, csrc/common.cuh) among the n_patch keys of its record is < k, ties broken by
 *      the lower index: exactly k masked patches per record.  `site` keeps the keys apart from the dropout sites
 *      (0 .. 4*depth).  mask: uint8 [B, n_patch]; counts: int32 [B], the masked patches of every record.
 *      seed == NULL: `mask` already holds a caller-supplied mask (any count per record) and is only counted.
 *      One CTA per record, the keys in shared memory (n_patch <= 12000); O(n_patch^2) compares per record. */
int ecgvit_mpm_mask(const uint32_t *seed, int B, int n_patch, int k, int site, uint8_t *mask, int *counts,
                    void *stream);
/* tok[b,0,:] = cls + pos[0];  tok[b,1+w,:] = (mask[b*n_patch+w] ? mask_token : e[b*n_patch+w,:]) + pos[1+w]
 * (ecgvit_embed_assemble with masked patches replaced by the learned token; dropout / dtype as there) */
int ecgvit_embed_assemble_masked(const void *e, const float *cls, const float *pos, const float *mask_token,
                                 const uint8_t *mask, void *tok, int B, int n_patch, int d, float dropout_p,
                                 int dropout_stream, const uint32_t *dropout_seed, int dtype, void *stream);
/* backward of the above: de = g[:,1:,:] on visible rows and 0 on masked rows; dpos += sum_b g; dcls += sum_b g[:,0];
 * dbias += sum over visible rows; dmask_token += sum over masked rows */
int ecgvit_embed_assemble_masked_bwd(const void *dtok, const uint8_t *mask, void *de, float *dcls, float *dpos,
                                     float *dbias, float *dmask_token, int B, int n_patch, int d, float dropout_p,
                                     int dropout_stream, const uint32_t *dropout_seed, int dtype, void *stream);
/* LayerNorm over the PATCH rows of a token matrix tok [B*(n_patch+1), d]: y[b*n_patch+w] = LN(tok[b*(n_patch+1)+1+w]);
 * y, mean and rstd are compact ([B*n_patch, d], [B*n_patch]).  dtype ECGVIT_BF16_RES32: tok is fp32, y bf16. */
int ecgvit_layernorm_patch_fwd(const void *tok, const float *gamma, const float *beta, void *y, float *mean,
                               float *rstd, int B, int n_patch, int d, float eps, int dtype, void *stream);
/* its backward: dtok (token-shaped, dtype of dy) is FULLY written: LN'(dy) on the patch rows, zeros on the CLS rows;
 * dgamma += ..; dbeta += ..; dcolsum (optional) += colsum(dtok).  scratch as for ecgvit_layernorm_bwd. */
int ecgvit_layernorm_patch_bwd(const void *dy, const void *tok, const float *gamma, const float *mean,
                               const float *rstd, void *dtok, float *dgamma, float *dbeta, float *dcolsum,
                               float *scratch, int B, int n_patch, int d, int dtype, void *stream);
/* Masked-patch MSE from the row partials of ECGVIT_EPI_BIAS_SUB_ROWSQ (rowsq fp32 [n_groups, B*n_patch]):
 *      count[0] = sum_b counts[b];  loss[0] = sum over masked rows, in a fixed order, of their partials / (count * K).
 *      One CTA: bit-identical from run to run.  count 0 gives NaN, as torch's mean over an empty selection. */
int ecgvit_mpm_loss(const float *rowsq, int n_groups, const uint8_t *mask, const int *counts, int B, int n_patch,
                    int K, float *loss, float *count, void *stream);
/* gradient of that loss w.r.t. the prediction: dpred = r * mask_row * 2 * grad_scale (* *grad_scale_dev) / (count * K)
 * for r [rows, ld] (dtype), mask [rows], count the device scalar written by ecgvit_mpm_loss; no host sync */
int ecgvit_mpm_dpred(const void *r, const uint8_t *mask, const float *count, int rows, int ld, int K,
                     float grad_scale, const float *grad_scale_dev, void *dpred, int dtype, void *stream);
/* reconstruction = r + target as fp32 [rows, K] (r, target: [rows, ld] in dtype).  In bf16 mode r is the stored bf16
 * residual, so this is bf16(pred - target) + target: an inspection output, not the exact prediction. */
int ecgvit_mpm_reconstruction(const void *r, const void *target, float *out, int rows, int ld, int K, int dtype,
                              void *stream);

/* ---- MAE-style pre-training (the encoder sees only the visible patches; a second, narrower block stack decodes).
 *      Added in ABI version 7 without changing any earlier entry point, so the version number stays 7.
 *
 *      Index build, one CTA per record (n_patch <= 12000): from mask uint8 [B, n_patch] (n_vis patches with mask 0 in
 *      every record) vis_idx int32 [B, n_vis] = the ascending positions of the visible patches, and slot int32
 *      [B, n_patch] = a patch's index among them, or -1 when it is masked. */
int ecgvit_mae_index(const uint8_t *mask, int B, int n_patch, int n_vis, int *vis_idx, int *slot, void *stream);
/* dst[b*n_dst + j, :] = src[b*n_src + idx[b*n_dst + j], :] for rows of ld elements (dtype BF16 / F32); the row length
 * must be a multiple of 16 bytes */
int ecgvit_row_gather(const void *src, void *dst, const int *idx, int B, int n_src, int n_dst, int ld, int dtype,
                      void *stream);
/* tok[b,0,:] = cls + pos[0];  tok[b,1+j,:] = e[b*n_vis+j,:] + pos[1 + vis_idx[b*n_vis+j]]; tok is [B*(n_vis+1), d].
 * Dropout (element index = position in tok) and dtype as ecgvit_embed_assemble. */
int ecgvit_embed_assemble_visible(const void *e, const float *cls, const float *pos, const int *vis_idx, void *tok,
                                  int B, int n_vis, int d, float dropout_p, int dropout_stream,
                                  const uint32_t *dropout_seed, int dtype, void *stream);
/* backward of the above (g = dropout mask applied to dtok): de = g[:,1:,:]; dcls += sum_b g[:,0]; dpos[0] += the same;
 * dpos[1+p] += sum over the records where patch p is visible of g[b, 1+slot[b,p]]; dbias += sum_{b,j} g[:,1:].
 * scratch: fp32 [n_patch, d].  Every sum runs in a fixed record order without float atomics: bit-identical from launch
 * to launch.  Three kernels: the position sums, then a two-pass fixed-order fold of them. */
int ecgvit_embed_assemble_visible_bwd(const void *dtok, const int *slot, void *de, float *dcls, float *dpos,
                                      float *dbias, float *scratch, int B, int n_patch, int n_vis, int d,
                                      float dropout_p, int dropout_stream, const uint32_t *dropout_seed, int dtype,
                                      void *stream);
/* decoder input u [B*(n_patch+1), d] from the embedded encoder output t [B*(n_vis+1), d]:
 * u[b,0] = t[b,0] + pos[0];  u[b,1+p] = (slot[b,p] >= 0 ? t[b, 1+slot[b,p]] : mask_token) + pos[1+p].
 * dtype ECGVIT_BF16_RES32: t bf16, u fp32. */
int ecgvit_mae_unshuffle(const void *t, const float *mask_token, const float *pos, const int *slot, void *u, int B,
                         int n_patch, int n_vis, int d, int dtype, void *stream);
/* its backward: dt (fully written) = the rows of du that t fed; dpos += sum_b du; dmask_token += sum of the masked rows.
 * scratch: fp32 [n_patch, d].  Fixed record order, no float atomics; three kernels, as the visible-assemble backward. */
int ecgvit_mae_unshuffle_bwd(const void *du, const int *slot, void *dt, float *dpos, float *dmask_token,
                             float *scratch, int B, int n_patch, int n_vis, int d, int dtype, void *stream);

/* ---- nn.LayerNorm(d, eps) forward (PreNorm.norm / mlp_head[0]); saves per-row mean and rstd (fp32) */
int ecgvit_layernorm_fwd(const void *x, const float *gamma, const float *beta, void *y, float *mean,
                         float *rstd, int M, int d, float eps, int dtype, void *stream);
/* backward: dx = (dres ? dres : 0) + LN'(dy); dgamma += ..; dbeta += ..
 * Without dropout (dxm NULL or p = 0): if dcolsum: dcolsum += colsum(dx).
 * With dropout (dx feeds a Linear through nn.Dropout, see "dropout" below): dxm = mask * dx / (1 - p) is written as
 * well and dcolsum += colsum(dxm).
 * scratch: fp32 workspace of ecgvit_layernorm_bwd_scratch_floats(d) elements (per-CTA column partials) */
int64_t ecgvit_layernorm_bwd_scratch_floats(int d);
/* defer_finalize != 0: only the per-CTA partial rows are written to `scratch`; the caller folds them into dgamma /
 * dbeta / dcolsum later with ecgvit_layernorm_bwd_finalize (e.g. on another stream, off the critical chain) and must
 * not reuse `scratch` before that has run. */
int ecgvit_layernorm_bwd(const void *dy, const void *x, const float *gamma, const float *mean,
                         const float *rstd, const void *dres, void *dx, float *dgamma, float *dbeta,
                         float *dcolsum, float *scratch, void *dxm, float dropout_p, int dropout_stream,
                         const uint32_t *dropout_seed, int M, int d, int defer_finalize, int dtype, void *stream);
int ecgvit_layernorm_bwd_finalize(const float *scratch, float *dgamma, float *dbeta, float *dcolsum, int M, int d,
                                  void *stream);
/* ecgvit_layernorm_bwd when dx feeds a Linear through element dropout (p >= 0) and drop path (see ecgvit_gemm_drop_path):
 * dxm = s[row / rows_per_record] * mask * dx (mask all ones when dropout_p = 0; fp32 before rounding) is written, dxm
 * must not be NULL, and dcolsum += colsum(dxm). */
int ecgvit_layernorm_bwd_drop_path(const void *dy, const void *x, const float *gamma, const float *mean,
                                   const float *rstd, const void *dres, void *dx, float *dgamma, float *dbeta,
                                   float *dcolsum, float *scratch, void *dxm, float dropout_p, int dropout_stream,
                                   const uint32_t *dropout_seed, int M, int d, int defer_finalize, int dtype,
                                   float path_p, int path_stream, int rows_per_record, void *stream);

/* ---- dense contraction  C[m,n] = sum_k A(m,k) * B(n,k)  with fused epilogue.
 *      Replaces nn.Linear forward / its autograd dgrad / wgrad (vit_pytorch Attention.to_qkv, to_out[0],
 *      FeedForward.net[0], net[3], ViT.to_patch_embedding[1]).
 *      a_kmajor=1: A stored row-major [M, K] with leading dimension lda (elements); 0: stored [K, M].
 *      b_kmajor=1: B stored row-major [N, K] with leading dimension ldb;            0: stored [K, N].
 *      dtype BF16 runs on tcgen05 (TMA-fed, TMEM accumulators); F32 runs on FFMA (parity mode). */
typedef struct ecgvit_gemm_args {
    int M, N, K;
    const void *A;
    int64_t lda;
    int a_kmajor;
    const void *B;
    int64_t ldb;
    int b_kmajor;
    int epilogue;       /* ECGVIT_EPI_* */
    void *out;
    int64_t ldo;
    void *out2;         /* BIAS_GELU: gelu output (same ld as out) */
    const void *aux;    /* BIAS_RES: residual; DGELU: pre-activation (same ld as out) */
    const float *bias;  /* fp32 [N] or NULL */
    int dtype;
    int split_k;        /* >1 only with ECGVIT_EPI_ATOMIC_F32; 0 = choose */
    /* nn.Dropout fused into the epilogue (p = 0 or seed = NULL: off).  BIAS_RES: out = drop(acc + bias) + aux;
     * BIAS_GELU: out2 = drop(gelu(out)); DGELU: out = drop(acc) * gelu'(aux).  See "dropout" below. */
    int dropout_stream;
    float dropout_p;
    const uint32_t *dropout_seed;
} ecgvit_gemm_args;
int ecgvit_gemm(const ecgvit_gemm_args *g, void *stream);

/* ---- drop path (stochastic depth, timm's DropPath): a residual branch is kept or dropped per RECORD.
 *      Added in ABI version 7 without changing any earlier entry point, so the version number stays 7.
 *
 *      Token row `row` of a [B * rows_per_record, d] matrix belongs to record b = row / rows_per_record, whose factor is
 *      s[b] = 1 / (1 - path_p) when the 16 bits of the dropout counter hash (see "dropout" below) that site `path_stream`
 *      assigns to element index b are >= round(path_p * 65536), else 0.  The rate is therefore quantised to a multiple of
 *      1/65536, as dropout's is.  The seed is the dropout seed of the call (g->dropout_seed / dropout_seed), which must
 *      be set when path_p > 0 even if dropout_p = 0 (element dropout off).  path_p = 0 makes every call below exactly its
 *      plain counterpart.  path_p outside [0, 1) and rows_per_record <= 0 are rejected before any launch.
 *
 *      GEMM: only with ECGVIT_EPI_BIAS_RES / ECGVIT_EPI_BIAS_RES_F32 (K-major A and B): out = s[row / rows_per_record] *
 *      drop(acc + bias) + aux.  Other epilogues with path_p > 0 are rejected. */
int ecgvit_gemm_drop_path(const ecgvit_gemm_args *g, float path_p, int path_stream, int rows_per_record, void *stream);

/* ---- softmax attention on the packed projection: replaces chunk(3) + rearrange + q k^T * scale +
 *      Softmax + attn v + rearrange back (vit_pytorch Attention.forward).
 *      qkv [B*N, 3*H*dh] (q | k | v, each head-major), o [B*N, H*dh], lse [B, H, N] fp32. */
int ecgvit_attention_fwd(const void *qkv, void *o, float *lse, int B, int N, int H, int dh, float scale,
                         float dropout_p, int dropout_stream, const uint32_t *dropout_seed, int dtype,
                         void *stream);
/* scratch: fp32 workspace of ecgvit_attention_bwd_scratch_floats(...) elements (rowsum(dO * O) of the tiled kernels
 * that serve N > 64 in bf16; 0 -> may be NULL) */
int64_t ecgvit_attention_bwd_scratch_floats(int B, int N, int H, int dh, int dtype);
int ecgvit_attention_bwd(const void *qkv, const void *o, const void *d_o, const float *lse, void *dqkv,
                         float *scratch, int B, int N, int H, int dh, float scale, float dropout_p,
                         int dropout_stream, const uint32_t *dropout_seed, int dtype, void *stream);

/* slow path for vit_pytorch's Recorder / the reference's EcgVitVisualizer (ecg_vit.py:176-193): the softmax
 * probabilities of one layer, fp32, probs[b * batch_stride + (h * N + i) * N + j] (no dropout: Recorder hooks
 * `attend`, the Softmax itself).  batch_stride >= H*N*N lets a [B, layers, H, N, N] tensor be filled layer by layer. */
int ecgvit_attention_probs(const void *qkv, float *probs, int B, int N, int H, int dh, float scale,
                           int64_t batch_stride, int dtype, void *stream);

/* ---- CLS pool + mlp_head (LayerNorm + Linear(d -> n_class)) + nn.BCEWithLogitsLoss (ecg_vit.py:118,144-148).
 *      tok [B*N, d]; logits fp32 [B, n_class]; loss: scalar (mean / sum) or [B, n_class] (none).
 *      labels may be NULL (logits only).  xn/mean/rstd are saved for backward.
 *      loss_weight: NULL, or the reference's `EcgVit.loss_weight` table (device fp32[n_weight]): element (b, k) of
 *      the loss is multiplied by loss_weight[(long)labels[b, k]] (ecg_vit.py:144-147 `weight[labels.long()]`; the
 *      index is clamped to the table, where torch would raise); 'mean' still divides by B * n_class. */
int ecgvit_head_fwd(const void *tok, const float *gamma, const float *beta, const float *w, const float *b,
                    const float *labels, const float *loss_weight, int n_weight, float *xn, float *mean,
                    float *rstd, float *logits, float *loss, int B, int N, int d, int n_class, int reduction,
                    float eps, int dtype, void *stream);
/* backward for reduction mean|sum with upstream gradient `grad_scale` (a host scalar, normally 1) times, when
 * `grad_scale_dev` is not NULL, the DEVICE scalar it points to (autograd's grad_output, read without a host sync):
 *      dlogits = grad_scale * weight * (sigmoid(z) - y) [/ (B*n_class)];  dw += ..; db += ..; dgamma/dbeta += ..;
 *      dtok is FULLY written: LN' rows at the CLS positions, zeros elsewhere; dcolsum += sum_b dtok[b,0,:] */
int ecgvit_head_bwd(const void *tok, const float *gamma, const float *w, const float *labels,
                    const float *loss_weight, int n_weight, const float *xn, const float *mean,
                    const float *rstd, const float *logits, void *dtok, float *dw, float *db, float *dgamma,
                    float *dbeta, float *dcolsum, float *scratch, int B, int N, int d, int n_class, int reduction,
                    float grad_scale, const float *grad_scale_dev, int dtype, void *stream);

/* ---- mean pool of vit_pytorch's ViT(pool='mean'): out[b, :] = mean over all N tokens (CLS included) of tok[b, :, :].
 *      tok [B*N, d] in the stream dtype (ECGVIT_BF16_RES32: fp32 tokens); out fp32 [B, d].  Each column is summed in
 *      a fixed order without atomics: bit-identical from run to run.  The pooled rows feed ecgvit_head_fwd /
 *      ecgvit_head_bwd as fp32 tokens with N = 1; the head's dcolsum is then sum_b dpool[b, :], the column sum of the
 *      broadcast gradient. */
int ecgvit_token_mean(const void *tok, float *out, int B, int N, int d, int dtype, void *stream);
/* its backward: dtok[b, t, :] = dpool[b, :] / N for every token t (dtok is FULLY written; bf16 in both bf16 modes) */
int ecgvit_token_mean_bwd(const float *dpool, void *dtok, int B, int N, int d, int dtype, void *stream);

/* ---- evaluation metrics on the device (SURVEY 8f rank 2): replaces the sklearn calls of
 *      ecg_transformer/util/train.py:12-56 `get_accuracy(preds, labels)`.
 *      preds (probabilities, fp32) and labels (multi-hot fp32) are [n_rows, n_class] device arrays.
 *      out (device double[6 + n_class]): [0] binary_accuracy, [1] weighted_binary_accuracy,
 *      [2] binary_negative_recall, [3] binary_positive_recall (names AND the swapped y_true / y_pred of
 *      util/train.py:47-55 kept), [4] macro_auc over the classes that have both labels (NaN if none),
 *      [5] how many such classes, [6 + c] AUROC of class c (NaN when undefined).  AUROC = exact integer
 *      Mann-Whitney count (ties 1/2) / (n+ n-), what sklearn's roc_auc_score evaluates to.
 *      scratch: ecgvit_eval_metrics_scratch_bytes(n_class) bytes of device memory (zeroed by the call). */
int64_t ecgvit_eval_metrics_scratch_bytes(int n_class);
int ecgvit_eval_metrics(const float *preds, const float *labels, int64_t n_rows, int n_class, int with_auc,
                        void *scratch, double *out, void *stream);

/* ---- dropout (nn.Dropout at the 5 sites per block + embedding of vit_pytorch; p wiring in ecg_vit.py:113-114).
 *      Counter-based: element `idx` of site `dropout_stream` is kept iff the 16 bits that hash(seed, stream,
 *      idx >> 1) (two 32x32->64 multiply-and-fold rounds, csrc/common.cuh) assigns to it are >= round(p * 65536); kept values are scaled by 1 / (1 - p).  `dropout_seed` points to
 *      a DEVICE uint32 the host refreshes every step, so forward and backward regenerate the same mask and no mask is
 *      stored.  Element indices: row * ld + col for [M, ld] tensors; ((b*H + h) * Np + query) * Np + key with
 *      Np = N rounded up to 64 for attention probabilities.
 *      Backward of a dropout that sits between a Linear and the residual add (to_out[1], net[4]):
 *      dym = mask * dy / (1 - p) (operand of the Linear's dgrad / wgrad), dcolsum += colsum(dym) (its bias gradient). */
int ecgvit_dropout_bwd_copy(const void *dy, void *dym, float *dcolsum, int M, int N, int64_t ld, float dropout_p,
                            int dropout_stream, const uint32_t *dropout_seed, int dtype, void *stream);
/* the same copy with drop path (see ecgvit_gemm_drop_path): dym = s[row / rows_per_record] * mask * dy; dropout_p may be 0 */
int ecgvit_dropout_bwd_copy_drop_path(const void *dy, void *dym, float *dcolsum, int M, int N, int64_t ld,
                                      float dropout_p, int dropout_stream, const uint32_t *dropout_seed, int dtype,
                                      float path_p, int path_stream, int rows_per_record, void *stream);

/* ---- column sum  out[n] += sum_m x[m, n]   (bias gradients) */
int ecgvit_colsum(const void *x, float *out, int M, int N, int64_t ld, int dtype, void *stream);

/* ---- nn.utils.clip_grad_norm_ (train.py:281) + torch.optim.AdamW.step (train.py:242-244,282) on flat
 *      fp32 buffers.  hyper (device, fp32[16]):
 *        [0] lr  [1] beta1  [2] beta2  [3] eps  [4] weight_decay  [5] 1-beta1^t  [6] 1-beta2^t
 *        [7] max_grad_norm (<=0: no clipping)  [8] grad_scale (1/world for DDP sum-allreduce)
 *        [9] 1-beta1  [10] 1-beta2  [11] 1-lr*weight_decay  [12] lr/(1-beta1^t)  [13] sqrt(1-beta2^t)
 *        ([9..13] are derived by the host in double precision, as torch.optim.AdamW derives them)
 *        [14] skip: non-zero makes ecgvit_adamw_step a no-op
 *        [15] 1 - d_t, the averaging rate of ecgvit_adamw_step_ema (derived by the host in double precision: 1 minus
 *             fp32(0.9999) in fp32 is 1.7e-4 off relative); unused by every other entry point
 *      stats (device, fp32[ECGVIT_STATS_FLOATS]): [0] sum of squares of (grad_scale*g)  [1] non-finite flag
 *        [2] total_norm (written by grad_sumsq, adamw and grad_scale_by_clip)  [3] updates SKIPPED because the norm was non-finite
 *        (incremented by adamw, never cleared by the library: `error_if_nonfinite` for a host that polls every k steps)
 *        [4..] per-CTA partials (scratch).
 *      The norm is reduced without atomics, so it is bit-identical on every replica and from run to run. */
#define ECGVIT_STATS_FLOATS 2052
/* `g` is the flat gradient buffer in `grad_dtype`: ECGVIT_F32, or ECGVIT_BF16 when a data-parallel run all-reduced the
 * gradients in bf16 (half the NVLink bytes; the moments and parameters stay fp32 either way). */
int ecgvit_grad_sumsq(const void *g, int grad_dtype, int64_t n, const float *hyper, float *stats, void *stream);
/* The same norm over the 64-element blocks whose id in group_map (device uint8[n / 64], the map of
 * ecgvit_adamw_step_grouped) is not 255: frozen parameters and parameters in no group do not count.  n must be a
 * multiple of 64; a slice offsets group_map by its first element / 64.  Same partials, finalize and determinism. */
int ecgvit_grad_sumsq_grouped(const void *g, int grad_dtype, int64_t n, const uint8_t *group_map, const float *hyper,
                              float *stats, void *stream);
/* The same norm, slice by slice: every call reduces one slice of the gradient buffer into its own `n_blocks` partial
 * slots [first_block, first_block + n_blocks) of the stats scratch (2048 slots in all) and may run as soon as that slice
 * is final -- e.g. per layer beside the rest of backward -- in any order and on any stream; ecgvit_grad_sumsq_finalize
 * then folds slots [0, n_blocks) in a fixed order into stats[0..2].  Deterministic for a fixed slicing. */
int ecgvit_grad_sumsq_partial(const void *g, int grad_dtype, int64_t n, const float *hyper, float *stats,
                              int first_block, int n_blocks, void *stream);
int ecgvit_grad_sumsq_finalize(float *stats, int n_blocks, void *stream);
/* flags: 0 for a whole-buffer update.  ECGVIT_ADAMW_SLICE: the call updates one slice (p, m, v, g, shadow all offset
 * alike) of the flat buffers; the slices of one update may be issued in any order and beside other kernels
 * (short-lived CTAs); exactly one of them carries ECGVIT_ADAMW_FIRST_SLICE and records the norm / the skipped-update
 * count.  hyper[14] != 0 turns the call into a no-op (a deferred-update slot with nothing pending). */
#define ECGVIT_ADAMW_SLICE 1
#define ECGVIT_ADAMW_FIRST_SLICE 2
int ecgvit_adamw_step(float *p, float *m, float *v, const void *g, int grad_dtype, void *shadow_bf16, int64_t n,
                      const float *hyper, float *stats, int flags, void *stream);
/* ecgvit_adamw_step with per-parameter-group learning rate and weight decay (layer-wise LR decay, no-decay sets).
 *      group_map (device uint8[n / 64]): the group id of every 64-element block of the flat buffers (every tensor
 *      starts on a 64-element boundary); id 255 leaves p, m, v and the shadow untouched (parameters in no group).
 *      group_table (device fp32[2 * n_groups], n_groups <= 255): [2i] = 1 - lr_i * weight_decay_i,
 *      [2i + 1] = lr_i / (1 - beta1^t), derived by the host in double precision; they replace hyper[11] / hyper[12].
 *      Everything else of hyper and stats (betas, eps, clipping, skip, the skipped-update counter) and the flags are
 *      those of ecgvit_adamw_step.  A slice offsets group_map by its first element / 64 (n must be a multiple of 64). */
int ecgvit_adamw_step_grouped(float *p, float *m, float *v, const void *g, int grad_dtype, void *shadow_bf16, int64_t n,
                              const uint8_t *group_map, const float *group_table, const float *hyper, float *stats,
                              int flags, void *stream);
/* ecgvit_adamw_step (group_map NULL) or ecgvit_adamw_step_grouped (group_map and group_table given; n a multiple of
 * 64) followed, per element the update writes, by the weight moving average
 *      ema = ema + hyper[15] * (p_new - ema)          (ema: device fp32[n], 16-byte aligned, offset like p by a slice)
 * computed from the p it has just written.  Same flags, hyper, stats and validation as those two entry points; what
 * they leave untouched (hyper[14] skip, a non-finite norm, group id 255) keeps its ema value too.
 *      Added in ABI version 7 without changing any earlier entry point, so the version number stays 7. */
int ecgvit_adamw_step_ema(float *p, float *m, float *v, const void *g, int grad_dtype, void *shadow_bf16, float *ema,
                          int64_t n, const uint8_t *group_map, const float *group_table, const float *hyper,
                          float *stats, int flags, void *stream);
/* in-place  g *= clip_coef  for API-compatible clip_grad_norm_ on a flat buffer */
int ecgvit_grad_scale_by_clip(float *g, int64_t n, const float *hyper, float *stats, void *stream);

/* ---- fp32 -> bf16 cast of a flat buffer (weight shadows) */
int ecgvit_cast_f32_to_bf16(const float *src, void *dst, int64_t n, void *stream);
/* a <-> b in place over n floats and, when shadow_bf16 is not NULL, shadow = bf16(new a) with the rounding of
 * ecgvit_cast_f32_to_bf16 (one pass, no temporary: swaps the master weights with their moving average, shadow
 * included; a second call restores all three bit for bit).  a, b and the shadow must be 16-byte aligned.
 *      Added in ABI version 7 without changing any earlier entry point, so the version number stays 7. */
int ecgvit_swap_f32_cast(float *a, float *b, void *shadow_bf16, int64_t n, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* ECGVIT_B200_H */
