/* libcfp — C ABI of the B200-native CFP fusion + cross-zone propagation path.
 *
 * The reference (denyingmxd/CFPNet) is pure PyTorch and has no FFI of its own;
 * this header is the boundary a maintainer binds with ctypes from the
 * reference's `src/models` modules (see INTEGRATION.md).  Each entry point
 * names the reference code it replaces (paths relative to the reference root).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer owned by the caller (PyTorch); the
 *     library borrows it for the duration of the enqueue, allocates nothing
 *     persistent and never synchronises the device;
 *   - work is enqueued on `stream` (a cudaStream_t passed as void*) of the
 *     caller's current device; the library is re-entrant (no global mutable
 *     state; the last error message is thread-local);
 *   - activations are token-major [B, N=H*W, C] unless stated otherwise;
 *     `dtype` selects the activation element type (CFP_F32 or CFP_BF16);
 *     packed weights are always fp32 in the layouts documented per struct;
 *   - return value 0 = enqueued; non-zero = rejected, message in
 *     cfp_last_error().  Unsupported (C, kernel size, dtype) combinations are
 *     hard errors: there is no fallback path.
 */
#ifndef CFP_H_
#define CFP_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CFP_ABI_VERSION 16

#if defined(__GNUC__)
#define CFP_API __attribute__((visibility("default")))
#else
#define CFP_API
#endif

enum cfp_dtype { CFP_F32 = 0, CFP_BF16 = 1 };

/* Per-level zone geometry: the host integers TransformerFusion.forward derives
 * from patch_info (src/models/fusion.py:67-84) plus the clipped in-image zone
 * rectangle of fusion.py:104.  Computed by cfpnet_b200.geometry.zone_geometry. */
typedef struct cfp_geom {
    int32_t zone_num;            /* zones per side (8)                                  */
    int32_t pad_h, pad_w;        /* F.pad amounts, fusion.py:136                        */
    int32_t p1, p2;              /* patch cells per zone                                */
    int32_t sy_wo, sx_wo, ey_wo, ex_wo; /* zone canvas in un-padded map coordinates     */
    int32_t tzh, tzw;            /* canvas size = ey-sy, ex-sx                          */
    int32_t interpolate;         /* canvas != zone_num*p -> bilinear resize branch      */
    int32_t ry0, ry1, rx0, rx1;  /* in-image zone rectangle (zone_mask), rows/cols      */
} cfp_geom;

/* One LoFTREncoderLayer (src/models/transformer.py:14-71), packed:
 *   wq_t [C][C], wkv_t [C][2C] (k_proj | v_proj), wm_t [C][C], w1_t [2C][2C],
 *   w2_t [2C][C]: nn.Linear weights transposed to [in][out];
 *   ln1_g/b, ln2_g/b [C].  DAPM uses only wq_t and wkv_t. */
typedef struct cfp_loftr_w {
    const float *wq_t, *wkv_t, *wm_t, *w1_t, *w2_t;
    const float *ln1_g, *ln1_b, *ln2_g, *ln2_b;
    /* bf16 tensor-core path: the chain's weights as eight [C x C] bf16 blocks in the canonical
     * K-major UMMA layout ([C/8][C][8] each), in consumption order: Wq, Wm, W1[:C,:C], W1[:C,C:],
     * W1[C:,:C], W1[C:,C:], W2[:,:C], W2[:,C:] (rows = outputs).  DAPM uses only the first block.
     * Required for CFP_BF16.  kv_tc: the k_proj and v_proj weights as two such blocks. */
    const void *tc, *kv_tc;
} cfp_loftr_w;

/* DAPM convs (transformer.py:197-200, 239-244) with eval-mode BN folded:
 *   conv1_t [(tap,cin<2C)][C], conv2_t [(tap,cin<C)][C]  (tap = ky*3+kx),
 *   weights pre-multiplied by the BN scale; shift1/shift2 [C]. */
typedef struct cfp_dapm_w {
    cfp_loftr_w attn;
    const float *conv1_t, *shift1, *conv2_t, *shift2;
    /* bf16 tensor-core path: the same (scaled) weights as bf16 blocks in the canonical K-major
     * UMMA layout, one [C/8][C][8] block per (source, tap): conv1_pk [2*9] blocks (source 0 =
     * feat0 channels, source 1 = message channels), conv2_pk [9] blocks.  Required for CFP_BF16. */
    const void *conv1_pk, *conv2_pk;
} cfp_dapm_w;

/* LKPM Block14 (src/models/convnext.py:42-58), eval-mode BN folded:
 *   dw_t [k*k][C] depthwise taps (tap = ky*k+kx) times BN scale, dw_shift [C];
 *   ln_g/b [C]; pw1_t [C][4C], pw1_b [4C]; pw2_t [4C][C], pw2_b [C]. */
typedef struct cfp_lkpm_w {
    const float *dw_t, *dw_shift, *ln_g, *ln_b, *pw1_t, *pw1_b, *pw2_t, *pw2_b;
    /* bf16 tensor-core path: the 4C hidden dim in 128-wide slices j (4C/128 of them); per slice two 16-bit blocks in
     * the canonical K-major UMMA layout ([K/8][N][8]), in consumption order W1_0, W2_0, W1_1, ..., each padded to
     * max(128*(C+16), C*144)*2 bytes:
     *   W1_j  bf16 [N=128][K=C+16]: (pwconv1.weight * ln_g)[128j:128(j+1), :], then one K step whose first column is
     *         (pwconv1.bias + pwconv1.weight @ ln_b)[128j:128(j+1)] (LayerNorm affine and bias folded in);
     *   W2_j  fp16 [N=C][K=128+16]: pwconv2.weight[:, 128j:128(j+1)], then one K step whose first column is
     *         pwconv2.bias for j = 0 and zero otherwise.
     * Required for CFP_BF16. */
    const void *tc;
    /* bf16 tensor-core depthwise conv: banded-Toeplitz blocks T_dy[n][kk] = dw_t-tap(dy, kk-n) (0 outside
     * 0 <= kk-n < k), n < 32, kk < 16*KS, KS = ceil((31+k)/16).  Vertical taps are grouped dy = 4a + b
     * (a < NA = ceil(k/4); zero blocks for dy >= k) with the four b's side by side along N:
     * bf16 [C][NA][KS][2][128 = b*32+n][8]  (per (a, k-step) one UMMA B block [2][128][8]).
     * Required for CFP_BF16 when k >= 15. */
    const void *dw_toep;
    int32_t ksize;
} cfp_lkpm_w;

/* TwinsTransformer (transformer.py:154-165): LSA layer, GSA layer, and the GSA
 * sub-sampling conv sr_t [(dy,dx,cin)][C] + sr_b [C] + LayerNorm srln_g/b [C]. */
typedef struct cfp_twins_w {
    cfp_loftr_w lsa, gsa;
    const float *sr_t, *sr_b, *srln_g, *srln_b;
    /* bf16 tensor-core path: one [C x C] bf16 UMMA block per tap (dy*ws+dx) of the sr conv. */
    const void *sr_tc;
    int32_t ws;
} cfp_twins_w;

/* HistogramEncoder (src/models/encoder.py:6-50): 9 pointwise stages with
 * eval-mode BN folded; w_t[i] is [Cin][Cout], b[i] is [Cout]. */
typedef struct cfp_hist_w {
    const float *w_t[9];
    const float *b[9];
    /* bf16 tensor-core path: stages 1..8 as bf16 UMMA blocks [Cin/8][Cout][8], concatenated in stage order
     * (106496 bytes); stage 0 (Cin = 1) uses w_t[0] / b[0]. */
    const void *tc;
} cfp_hist_w;

CFP_API int cfp_version(void);
/* Thread-local message of the last failed call ("" if none). */
CFP_API const char *cfp_last_error(void);

/* Scratch bytes (fp32 attention state + token scratch) one fusion call needs;
 * the caller allocates it (torch.empty) and passes it to the layer calls.  The
 * size covers every entry point of the level: those that take the geometry
 * (zone_num^2 zones) and those that do not (laid out for 64 zones). */
CFP_API size_t cfp_workspace_bytes(int B, int H, int W, int C, int ws, int large_kernel, int dtype,
                                   const cfp_geom *g);

/* a2. Zone geometry of one TransformerFusion call, host arithmetic only (no device work, no stream).
 * Replaces patch_info_from_rect_data (src/utils/dataloader.py:13-40: per-frame pad / patch / index
 * integers, hard-coded 480x640 canvas, float32 divisions truncated toward zero), the batch-wise max / min
 * of fusion.py:75-78 and the integer block of fusion.py:67-84,104.  rects [B][Z][4] float rows
 * (y0,x0,y1,x1) in pixels (host memory); max_width = max_resolution[1] of the level (160 / 80 / 40:
 * cell size 640/max_width px); H, W = the level's map.  Fills *out; non-zero return (+ message) for
 * layouts on which the reference's own forward is undefined (canvas slice outside the padded map,
 * in-image canvas cells != zone rectangle cells).  Bit-exact with the reference's integers on the 216
 * layouts of tests/golden/geometry_cases.json (tests/test_host.py). */
CFP_API int cfp_geometry_from_rects(const float *rects, int B, int Z, int max_width, int H, int W, cfp_geom *out);

/* a1. HistogramEncoder.forward (encoder.py:45-50; deltar.py:40).
 * hist [rows] fp32 zone depth samples (rows = B*Z*S) -> out32 [rows][32],
 * out64 [rows][64], out128 [rows][128] in `dtype`. */
CFP_API int cfp_hist_encoder_fwd(const float *hist, void *out32, void *out64, void *out128, int64_t rows,
                         const cfp_hist_w *w, int dtype, void *stream);

/* a3. The three masks TransformerFusion.forward materialises (fusion.py:103-120),
 * as bytes (0/1), without the channel repeat: zone_mask [B][H*W],
 * hist_mask [B*Z][p1*p2], pad_mask [B][tzh][tzw].  mask = [B][Z] validity bytes.
 * Export for the bit-exact tests; the layer kernels use cfp_geom directly. */
CFP_API int cfp_zone_masks(const uint8_t *mask, uint8_t *zone_mask, uint8_t *hist_mask, uint8_t *pad_mask,
                   int B, int H, int W, const cfp_geom *g, void *stream);

/* a4. Positional-encoding add + NCHW -> token-major (fusion.py:92-97):
 * tokens[b][y*W+x][c] = x[b][c][y][x] + pos[(oy+y)*pos_w + ox+x][c]; pos is the
 * [pos_h*pos_w][C] table (max_resolution).  The crop offsets come from one of two places:
 *   crop == NULL: (oy, ox) as passed; the crop must lie inside the table.
 *   crop != NULL: (oy, ox) = (crop[0], crop[1]), int32 in DEVICE memory, read when the kernel runs: a CUDA-graph replay of
 *     a forward then takes fresh offsets from the buffer instead of freezing the captured ones (the reference draws them
 *     per call, fusion.py:88-91).  The host cannot see these offsets and does not range-check them: the caller keeps
 *     0 <= crop[0] <= pos_h - H, 0 <= crop[1] <= pos_w - W.  The map must fit the table, and oy, ox must be 0. */
CFP_API int cfp_posenc_tokens_fwd(const void *x_nchw, const float *pos, void *tokens, int B, int C, int H,
                          int W, int pos_h, int pos_w, int oy, int ox, const int *crop, int dtype, void *stream);
/* fusion.py:186: token-major -> contiguous NCHW. */
CFP_API int cfp_tokens_to_nchw(const void *tokens, void *out_nchw, int B, int C, int H, int W, int dtype,
                       void *stream);

/* a5. `hist2image` branch (fusion.py:132-157 + transformer.py:41-71 +
 * attention.py:20-52).  feat0 [B][N][C] is updated in place; emb is the map the
 * zone canvas is cut from (== feat0 under --change_embedding).  zone_tok
 * [B*Z][S][C] are the raw histogram tokens (positional_encodings2 `pos2` [S][C]
 * is added inside); mask [B][Z] bytes.  assign != 0 = --no_skip_inside. */
CFP_API int cfp_d2i_fwd(void *feat0, const void *emb, const void *zone_tok, const float *pos2,
                const uint8_t *mask, int B, int H, int W, int C, int S, const cfp_geom *g,
                const cfp_loftr_w *w, int assign, void *workspace, size_t workspace_bytes,
                int dtype, void *stream);

/* a6. DAPM, LoFTREncoderLayer_newcross9.forward (transformer.py:204-248); in place. */
CFP_API int cfp_dapm_fwd(void *feat0, int B, int H, int W, int C, const cfp_geom *g, const cfp_dapm_w *w,
                 void *workspace, size_t workspace_bytes, int dtype, void *stream);

/* a7. LKPM, Block14.forward (convnext.py:42-58) on token-major maps; in place. */
CFP_API int cfp_lkpm_fwd(void *feat0, int B, int H, int W, int C, const cfp_lkpm_w *w, void *workspace,
                 size_t workspace_bytes, int dtype, void *stream);

/* a9. `image` layer, TwinsTransformer.forward (transformer.py:89-116, 138-150,
 * 160-165): LSA then GSA, 8 heads; in place. */
CFP_API int cfp_twins_fwd(void *feat0, int B, int H, int W, int C, const cfp_twins_w *w, void *workspace,
                  size_t workspace_bytes, int dtype, void *stream);
/* The same layer as the LAST layer of a TransformerFusion call: the GSA result is written to the caller's contiguous NCHW
 * map `out_nchw` (fusion.py:186, the rearrange back to 'b c h w') by the layer's last epilogue instead of going through
 * feat0 and cfp_tokens_to_nchw; feat0 holds the LSA result afterwards and is scratch. */
CFP_API int cfp_twins_nchw_fwd(void *feat0, void *out_nchw, int B, int H, int W, int C, const cfp_twins_w *w,
                       void *workspace, size_t workspace_bytes, int dtype, void *stream);

/* ---- Training step (BASELINE config 5; reference train.py:96-135 with the modules in .train() mode, BatchNorm on
 * batch statistics per replica as under nn.DataParallel, train.py:45).  The reference differentiates its modules with
 * autograd; here the step is a sequence of these fp32 building blocks (token-major [rows][C] maps), ordered by
 * cfpnet_b200/train.py exactly as oracle/cfp_oracle_bwd.py states the backward.  Each names the reference op it serves.
 *
 * cfp_tr_gemm: C[M][N] (+)= A . B (+ bias[N]); element (i,k) of A at a[i*a_rs + k*a_cs], (k,j) of B at b[k*b_rs + j*b_cs].
 *   nn.Linear / Conv1d(k=1) forward x W^T + b (encoder.py:19-23, convnext.py:51-53), its input gradient dy W and its
 *   weight gradient dy^T x (a reduction over every row of the batch: split over K across CTAs, fp32 atomics).
 *   accumulate != 0 adds to the existing C. */
CFP_API int cfp_tr_gemm(const float *a, int64_t a_rs, int64_t a_cs, const float *b, int64_t b_rs, int64_t b_cs, float *c,
                        int64_t c_rs, int M, int N, int K, const float *bias, int accumulate, void *stream);
/* out[c] = sum_r x[r][c]: bias gradients. */
CFP_API int cfp_tr_colsum(const float *x, float *out, int64_t rows, int C, void *stream);
/* Train-mode BatchNorm (encoder.py:21-23, convnext.py:45-46, transformer.py:239-244): batch mean and biased variance
 * over the rows (two passes), rstd = rsqrt(var + eps); running_mean / running_var (nullable) updated in place with
 * `momentum` and the unbiased variance, as torch.nn.functional.batch_norm does.  scratch: 2*C floats. */
CFP_API int cfp_tr_bn_stats(const float *x, int64_t rows, int C, float eps, float momentum, float *mean, float *rstd,
                            float *running_mean, float *running_var, float *scratch, void *stream);
/* y = (x - mean) * rstd * gamma + beta, then ReLU when relu != 0. */
CFP_API int cfp_tr_bn_apply(const float *x, const float *mean, const float *rstd, const float *gamma, const float *beta,
                            float *y, int64_t rows, int C, int relu, void *stream);
/* Backward of cfp_tr_bn_apply (+ the ReLU behind it when relu != 0) with batch statistics:
 * dx = gamma*rstd/n * (n g - sum g - xhat sum(g xhat)); dgamma = sum g xhat, dbeta = sum g. */
CFP_API int cfp_tr_bn_bwd(const float *dy, const float *x, const float *mean, const float *rstd, const float *gamma,
                          const float *beta, float *dx, float *dgamma, float *dbeta, int64_t rows, int C, int relu,
                          void *stream);
/* LayerNorm over the channel dim (convnext.py:60-85 channels_last, nn.LayerNorm of transformer.py:36-37) and its
 * backward (dx, dgamma, dbeta). */
CFP_API int cfp_tr_ln_fwd(const float *x, const float *g, const float *b, float *y, int64_t rows, int C, float eps,
                          void *stream);
CFP_API int cfp_tr_ln_bwd(const float *x, const float *g, const float *dy, float *dx, float *dg, float *db, int64_t rows,
                          int C, float eps, void *stream);
/* Elementwise: op 0 out = a + b | 1 out = a * (b > 0) | 2 out = gelu_erf(a) | 3 out = a * gelu_erf'(b) | 4 out = relu(a)
 * | 5 out = a * d/db(elu(b) + 1) | 6 out = elu(a) + 1 | 7 out = -a / b | 8 out = leaky_relu(a, 0.01) (nn.LeakyReLU() of
 * decoder.py) | 9 out = a * (b > 0 ? 1 : 0.01), its gradient. */
CFP_API int cfp_tr_ew(const float *a, const float *b, float *out, int64_t n, int op, void *stream);
/* ---- second slice of the training step: the linear-attention layers and the DAPM convolutions of a TransformerFusion
 * call in train mode (fusion.py:52-188, transformer.py:41-71,89-150,204-248, attention.py:31-49 under autograd in the
 * reference).  cfpnet_b200/train_seq.py orders these primitives (forward and the closed-form backward); every
 * regrouping of tokens is a gather / scatter-add over an int32 index vector built once on the host (-1 = a zero row).
 *
 * cfp_tr_gather_rows: out[i][:] = idx[i] >= 0 ? src[idx[i]][:] : 0 (zone canvas cells fusion.py:139-141, LSA windows
 *   transformer.py:94-104, DAPM inside / outside sets transformer.py:214-221, 3x3 conv taps, the sr conv's strided taps).
 * cfp_tr_scatter_add_rows: out = base (base_rows rows, copied unless out == base); out[idx[i]][:] += src[i][:] - the
 *   adjoint of the gather and the `feat0[zone_mask] += ...` of fusion.py:157. */
CFP_API int cfp_tr_gather_rows(const float *src, const int *idx, float *out, int64_t n, int C, void *stream);
CFP_API int cfp_tr_scatter_add_rows(const float *src, const int *idx, const float *base, float *out, int64_t n,
                                    int64_t base_rows, int C, void *stream);
/* Attention state of G groups of R rows, nh heads of d = C / nh channels (attention.py:39-44):
 *   kv[g][h][i][j] = sum_r a[g][r][h d + i] * b[g][r][h d + j];  as[g][c] = sum_r (w ? w[g][r][h(c)] : 1) * a[g][r][c].
 * Forward: a = elu(k)+1, b = v.  Backward: a = Q, b = dnum, w = dden (the state's gradient). */
CFP_API int cfp_tr_attn_reduce(const float *a, const float *b, const float *w, float *kv, float *as, int G, int R, int C,
                               int nh, void *stream);
/* out[g][r][h d + o] = sum_k x[g][r][h d + k] * (transpose ? kv[g][h][o][k] : kv[g][h][k][o])  (Q x KV and its adjoints). */
CFP_API int cfp_tr_attn_apply(const float *x, const float *kv, float *out, int G, int R, int C, int nh, int transpose,
                              void *stream);
/* out[row][h] = sum_k a[row][h d + k] * b[brow][h d + k] + eps, brow = rows_per_group ? row / rows_per_group : row
 * (the normaliser Q . Ksum + eps of attention.py:42; dmsg . msg in the backward). */
CFP_API int cfp_tr_head_dot(const float *a, const float *b, float *out, int64_t rows, int C, int nh, int rows_per_group,
                            float eps, void *stream);
/* Row arithmetic with a per-(row, head) operand s [rows][nh] or a per-group operand b indexed by row / rows_per_group:
 * op 0 out = a * s | 1 out = a / s | 2 out = a + s * b[group][c] | 3 out = a + b[group][c] | 4 out = a * b[group]
 * (b a vector: the zone mask of fusion.py:144).  out may alias a. */
CFP_API int cfp_tr_rowop(const float *a, const float *s, const float *b, float *out, int64_t rows, int C, int nh,
                         int rows_per_group, int op, void *stream);
/* k x k depthwise conv on a token-major map, out = conv(in) + shift[c] (ReLU when relu != 0): Block14.dwconv2 in train
 * mode (convnext.py:45; shift = the conv bias) and, with the taps flipped in both axes and shift = 0, its input
 * gradient.  taps_t [k*k][C]. */
CFP_API int cfp_tr_dwconv(const float *in, float *out, int B, int H, int W, int C, int ksize, const float *taps_t,
                          const float *shift, int relu, void *stream);
/* dw[c][i][j] = sum_{b,y,x} dy[b][y][x][c] * x[b][y+i-p][x+j-p][c]: weight gradient of that conv, [C][k][k]. */
CFP_API int cfp_tr_dwconv_wgrad(const float *x, const float *dy, float *dw, int B, int H, int W, int C, int ksize,
                                void *stream);

/* Optimizer step on the flat gradient bucket (train.py:124-129: clip_grad_norm_(parameters, 0.1), AdamW.step()).
 * cfp_tr_sumsq: out[0] = sum_i (x[i] * scale)^2 (the squared global gradient norm; scale = 1 / world after a sum
 * all-reduce).  `out` is CFP_SUMSQ_FLOATS floats, zero-initialised once by the caller (result, per-CTA partials, a
 * ticket): the sum is formed in a fixed order, so replicas that hold the same bucket get the same bits.  cfp_tr_adamw: torch.optim.AdamW's update of p / m / v [n] with gradient g * grad_scale * min(1, max_norm /
 * (sqrt(*sumsq) + 1e-6)) (max_norm <= 0: no clipping, sumsq may be NULL); `step` >= 1 is the bias-correction step count;
 * element i uses the learning rate seg_lr[s] of the segment with seg_end[s-1] <= i < seg_end[s] (device arrays [nseg]: the
 * reference's 1x / 10x parameter groups, train.py:75-76).  Nothing here synchronises with the host. */
#define CFP_SUMSQ_FLOATS 1026
CFP_API int cfp_tr_sumsq(const float *x, int64_t n, float scale, float *out, void *stream);
CFP_API int cfp_tr_adamw(float *p, const float *g, float *m, float *v, int64_t n, const int64_t *seg_end, const float *seg_lr,
                         int nseg, float beta1, float beta2, float eps, float weight_decay, int step, float grad_scale,
                         const float *sumsq, float max_norm, void *stream);

/* ---- Decoder shell (SURVEY.md 8 f1) and adaptive-bins head (f2) on channels-last maps [B][H][W][pitch] - the token-major
 * layout of the fusion path.  `dtype` selects the engine and the element type of the maps:
 *   CFP_BF16: bf16 maps, the convolutions and conv_out on the tensor cores (tcgen05); the channel counts, pitches and
 *     channel offsets of the channels-last maps are multiples of 8;
 *   CFP_F32: the exact fp32 engine: fp32 maps, fp32 FFMA with fp32 accumulation (no TF32 or bf16 operands), no atomics
 *     (every output is summed in one fixed order: two runs give the same bits); those counts are multiples of 4.
 *
 * cfp_conv_fwd: k x k convolution (k = 1, 3; stride 1, zero padding (k-1)/2) as an implicit GEMM:
 *   out[b][y][x][out_coff + o] = act(sum_{taps, c} in[b][y+dy][x+dx][c] w[o][c][dy][dx] + shift[o]), act = LeakyReLU with
 *   `leaky_slope` (1.0 = none).  Serves decoder.py:43-48 (conv3x3 + BatchNorm2d folded by the host + LeakyReLU, twice per
 *   UpSampleBN), :70,76-80 (1x1 / 3x3 convs with bias) and DepthRegression.conv3x3 (:13).  cout in {32, 64, 128, 256};
 *   shift [cout] fp32; out has pitch out_pitch (write into a slice of a wider buffer: torch.cat).
 *   CFP_BF16: cin: input channels, zero-padded to a multiple of 16 (= the input's pitch); kchunk (multiple of 16, divides
 *     cin, cout * kchunk <= 20480): channels per staged K-chunk; w: bf16 blocks [cin / kchunk][k * k][kchunk / 8][cout][8]
 *     (canonical K-major UMMA layout per (chunk, tap)).
 *   CFP_F32: cin is a multiple of 4 and equal to the input's pitch (no padding); kchunk must be 0 (no K-chunks); w is fp32
 *     [k * k][cin][cout] (tap = ky * k + kx).
 * cfp_upsample_concat: UpSampleBN's input (decoder.py:51-58): out [B][H][W][c_out] = [ bilinear(align_corners) resize of
 *   lo [B][h][w][c_lo] (pitch lo_pitch) | skip [B][c_skip][H][W] (fp32 NCHW, the image encoder's feature; any c_skip) | zeros ].
 * cfp_posenc_tokens_nhwc_fwd: cfp_posenc_tokens_fwd for a caller that already holds the map channels-last (pitch x_pitch):
 *   tokens = x + pos crop, with the same two sources of the crop offsets (crop == NULL: oy, ox, range-checked; crop !=
 *   NULL: device offsets the caller keeps inside the table, oy = ox = 0): a CUDA-graph replay of the decoder takes fresh
 *   offsets from the buffer.
 * cfp_copy_channels: dst[row][coff : coff + C] = src[row][0 : C] (pitches in elements).
 * cfp_head_bins: DepthRegression's regressor branch (decoder.py:24-36, norm 'linear') + the bin geometry of deltar.py:52-57:
 *   per-frame channel mean of x [B][npix][pitch] (E channels) -> conv1x1 (wc [E][E], no bias) -> Linear(E, hidden) ->
 *   LeakyReLU -> Linear(hidden, hidden) -> LeakyReLU -> Linear(hidden, n_bins) -> relu + 0.1 -> / sum -> edges [B][n_bins + 1]
 *   = cumsum([min_val, (max_val - min_val) y]), centres [B][n_bins].  Weights fp32 row-major [out][in]; mean_scratch [B][E].
 *   CFP_F32 forms the channel mean per frame in one CTA (no atomics); the regressor is the same for both engines.
 * cfp_head_expect: conv_out (1x1, E = 128 -> n_bins, bias) + softmax over the bins + sum_j p_j centre_j in one kernel:
 *   x [B][npix][pitch] (the range-attention maps), pred [B][npix] fp32; prob (nullable) [B][n_bins][npix] fp32 is the
 *   probability volume the reference returns in eval mode.  w is conv_out's [n_bins][128] weight: for CFP_BF16 the
 *   canonical UMMA block, for CFP_F32 transposed to fp32 [128][n_bins] (softmax with expf and true divisions). */
CFP_API int cfp_conv_fwd(const void *in, int B, int H, int W, int cin, int cout, int ksize, int kchunk, const void *w,
                         const float *shift, float leaky_slope, void *out, int out_pitch, int out_coff, int dtype, void *stream);
CFP_API int cfp_upsample_concat(const void *lo, int h, int w, int c_lo, int lo_pitch, const float *skip, int c_skip, void *out,
                                int B, int H, int W, int c_out, int dtype, void *stream);
CFP_API int cfp_posenc_tokens_nhwc_fwd(const void *x, int x_pitch, const float *pos, void *tokens, int B, int C, int H, int W,
                                       int pos_h, int pos_w, int oy, int ox, const int *crop, int dtype, void *stream);
CFP_API int cfp_copy_channels(const void *src, int src_pitch, void *dst, int dst_pitch, int coff, int C, int64_t rows, int dtype,
                              void *stream);
CFP_API int cfp_head_bins(const void *x, int pitch, int B, int npix, int E, const float *wc, const float *w0, const float *b0,
                          const float *w2, const float *b2, const float *w4, const float *b4, int hidden, int n_bins, float min_val,
                          float max_val, float *mean_scratch, float *edges, float *centres, int dtype, void *stream);
CFP_API int cfp_head_expect(const void *x, int pitch, int B, int npix, const void *w, const float *bias, const float *centres,
                            int n_bins, float *pred, float *prob, int dtype, void *stream);

/* ---- The decoder shell and head in train mode (reference train.py:96-135 differentiates decoder.py / deltar.py:50-61 with
 * autograd): the adjoints no forward kernel computes.  fp32 FFMA, no atomics, fixed summation order (two launches give the
 * same bits).  cfpnet_b200/decoder_train.py sequences them with the forward kernels above on the CFP_F32 engine: a conv's
 * input gradient is cfp_conv_fwd with the taps mirrored and in / out channels swapped.
 *
 * cfp_tr_conv_wgrad_f32: weight gradient of a k x k conv (k = 1, 3; stride 1, zero padding k / 2) on channels-last maps,
 *   dw[tap][ci][co] = sum_{b,y,x} x[b][y + ky - k/2][x + kx - k/2][ci] dy[b][y][x][co] (tap = ky k + kx: the fp32 weight
 *   layout of cfp_conv_fwd with CFP_F32).  cin, cout multiples of 4; x has pitch cin, dy pitch cout.  The B*H*W pixels are split
 *   into ranges, each writes a partial into `scratch`, a second pass adds them in range order:
 *   cfp_tr_conv_wgrad_scratch_floats(B, H, W, cin, cout, ksize) floats (pure host arithmetic; 0 = no scratch needed).
 * cfp_tr_upsample_concat_bwd_f32: adjoint of cfp_upsample_concat with CFP_F32.  dcat [B][H][W][pitch] -> d_lo [B][h][w][c_lo]
 *   (channels-last, the adjoint of the align_corners bilinear resize, gathered per low-resolution pixel) and d_skip
 *   [B][c_skip][H][W] (NCHW, channels c_lo .. c_lo + c_skip of dcat).
 * cfp_tr_head_expect_bwd_f32: adjoint of cfp_head_expect with CFP_F32 given its probability volume prob [B][n_bins][npix], pred
 *   [B][npix], centres [B][n_bins] and dpred [B][npix]: dlogit [B*npix][n_bins] = p (centre - pred) dpred, dcentres
 *   [B][n_bins] = sum_pixels p dpred.  scratch: B * ((npix + 31) / 32) * n_bins floats.
 * cfp_tr_head_bins_bwd_f32: one CTA per frame.  z [B][n_bins] = the regressor's output before relu + 0.1; d_edges [B][n_bins
 *   + 1] and d_centres [B][n_bins] (either nullable = zero) are the cotangents of cfp_head_bins's outputs -> dz. */
CFP_API size_t cfp_tr_conv_wgrad_scratch_floats(int B, int H, int W, int cin, int cout, int ksize);
CFP_API int cfp_tr_conv_wgrad_f32(const float *x, const float *dy, float *dw, float *scratch, int B, int H, int W, int cin, int cout,
                                  int ksize, void *stream);
CFP_API int cfp_tr_upsample_concat_bwd_f32(const float *dcat, int pitch, float *d_lo, int h, int w, int c_lo, float *d_skip, int c_skip,
                                           int B, int H, int W, void *stream);
CFP_API int cfp_tr_head_expect_bwd_f32(const float *prob, const float *pred, const float *centres, const float *dpred, int B, int npix,
                                       int n_bins, float *dlogit, float *dcentres, float *scratch, void *stream);
CFP_API int cfp_tr_head_bins_bwd_f32(const float *z, const float *d_edges, const float *d_centres, float *dz, int B, int n_bins,
                                     float min_val, float max_val, void *stream);

/* ---- Input side (SURVEY.md 8 f3; the reference runs these on the host CPU inside its dataloader, one frame at a time).
 *
 * cfp_zone_hist: get_hist_parallel (src/utils/dataloader.py:84-134) for a batch of depth maps dep [B][H][W] (metres):
 *   zone (zy, zx) of the zone_num x zone_num grid is the ph x pw patch at (sy + zy ph, sx + zx pw); its depths are binned
 *   like torch.histc(bins = nbins, min = 0, max = max_distance), bin 0 is cleared, 20 is subtracted from every count
 *   (clipped at 0), only the contiguous run of non-zero bins with the largest sum survives, and in float64
 *   mu = sum(centre count) / (n + 1e-9), sigma = sqrt(sum(count (centre - mu)^2) / (n + 1e-9)) + 1e-9.
 *   centres [nbins] (device, double) are the bin centres as the reference forms them (:120).  Outputs: fh [B][Z][2] =
 *   (mu, sigma) fp32, mask [B][Z] = n > 0, hist_out [B][Z][nbins] int32 (nullable) = the surviving counts.
 * cfp_zone_samples: sample_point_from_hist_parallel (:65-81): fh [zones][2], mask [zones] -> out [zones][S]; mode 0
 *   (sample_uniform): out = w0[s] (mu - 3 sigma) + w1[s] (mu + 3 sigma) with w0 / w1 [S] = the reference's two linspace
 *   ramps, every operation rounded to fp32 as the reference's (bit-identical results); mode 1: normal quantiles
 *   mu + sigma w0[s] sqrt(2), w0[s] = erfinv(2 ppf_s - 1).  Zones with mask == 0 give zeros. */
CFP_API int cfp_zone_hist(const float *dep, int B, int H, int W, int sy, int sx, int ph, int pw, int zone_num, int nbins,
                          float max_distance, const double *centres, float *fh, uint8_t *mask, int *hist_out, void *stream);
CFP_API int cfp_zone_samples(const float *fh, const uint8_t *mask, float *out, int64_t zones, int S, const float *w0,
                             const float *w1, int mode, void *stream);

/* ---- Loss and metrics (SURVEY.md 8 f4).
 * cfp_silog_fwd: SILogLoss.forward (src/loss.py:9-19): pred [B][1][h][w] is resized to the target [B][1][H][W] (bilinear,
 *   align_corners; interpolate == 0: same size, no resize), g = log(up) - log(target) over the pixels with mask != 0 (NULL:
 *   all), loss = 10 sqrt(var_unbiased(g) + 0.15 mean(g)^2).  Sums are accumulated in float64 in a fixed order.  scratch:
 *   CFP_SILOG_SCRATCH_DOUBLES doubles, zeroed once by the caller; afterwards scratch[0..3] = n, mean, D, loss (what
 *   cfp_silog_bwd reads).  cfp_silog_bwd: grad_pred [B][1][h][w] = grad_out * dloss/dpred (zeroed inside).
 * cfp_depth_metrics: compute_errors (src/utils/metrics.py:4-24) over the n-element maps gt / pred where valid != 0 (NULL:
 *   all): out[0..8] = a1 a2 a3 abs_rel rmse log_10 rmse_log silog sq_rel, out[9] = number of valid pixels (device doubles).
 *   scratch: CFP_METRICS_SCRATCH_DOUBLES doubles, zeroed once by the caller. */
#define CFP_SILOG_SCRATCH_DOUBLES 1544
#define CFP_METRICS_SCRATCH_DOUBLES 5634
CFP_API int cfp_silog_fwd(const float *pred, const float *target, const uint8_t *mask, int B, int h, int w, int H, int W,
                          int interpolate, double *scratch, float *loss, void *stream);
CFP_API int cfp_silog_bwd(const float *pred, const float *target, const uint8_t *mask, int B, int h, int w, int H, int W,
                          int interpolate, const double *scratch, float grad_out, float *grad_pred, void *stream);
CFP_API int cfp_depth_metrics(const float *gt, const float *pred, const uint8_t *valid, int64_t n, double *scratch, double *out,
                              void *stream);

/* Accounting / tracing (no reference counterpart: the reference has no profiling hooks,
 * SURVEY.md §5).  cfp_launch_count: kernels this process has enqueued since load (all threads: a training
 * step's backward is enqueued from autograd's thread).
 * cfp_profile_start: from now on one CUDA event is recorded per kernel launch on the call's stream (all threads).  cfp_profile_stop: waits for the recorded events (the one place the library
 * blocks), writes {"kernel_name": [launches, total_ms], ...} as JSON into out[cap]. */
CFP_API int64_t cfp_launch_count(void);
/* Programmatic dependent launch of the bf16-path kernels for the calling thread: 1 = on (the default: a kernel's
 * prologue overlaps the previous kernel's drain; measured -3.5 % on a single stream), 0 = off (what FusionPath selects
 * while it runs the three levels on three streams: pre-launched CTAs then only take slots from the other streams'
 * kernels, measured +1.5 %), -1 = back to the default.  Returns the previous setting.  CFP_NO_PDL=1 in the
 * environment disables it process-wide. */
CFP_API int cfp_set_pdl(int on);
/* Known-answer self-test of the tcgen05 engine (tests only): d[m][j] = sum_k a[m+row_shift][k] *
 * b[j][k] for m < 128; a [rows_a][k] and b [n][k] are bf16 row-major, d [128][n] fp32. */
CFP_API int cfp_selftest_umma(const void *a, const void *b, float *d, int rows_a, int n, int k, int row_shift,
                              void *stream);
CFP_API int cfp_profile_start(void);
CFP_API int cfp_profile_stop(char *out, size_t cap);

#ifdef __cplusplus
}
#endif
#endif /* CFP_H_ */
