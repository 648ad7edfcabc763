// Internal (C++) launch interface between cfp_api.cu and the kernel files.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>
#include "../../include/cfp.h"

namespace cfp {

// Workspace partition of one fusion call (all offsets in bytes, 256-aligned).
struct WsLayout {
    size_t kv, kv_bytes;        // fp32 attention state: [groups][C*dh] KV then [groups][C] Ksum
    size_t tok_a, tok_b;        // two token-major scratch maps [B][N][C] in the activation dtype
    size_t tok_bytes;
    size_t sr, sr_bytes;        // GSA sub-sampled tokens, fp32 [B][Ns][C]
    size_t canvas, canvas_bytes;  // hist2image resize branch: [B][zn*p1*zn*p2][C] activation dtype
    size_t planes, planes_bytes;  // bf16 LKPM: padded channel planes (UMMA layout) + planar output
    size_t total;
};
WsLayout ws_layout(int B, int H, int W, int C, int ws, int large_kernel, int dtype, const cfp_geom* g);

inline size_t elem_size(int dtype) { return dtype == CFP_F32 ? 4 : 2; }

// k_layout.cu
int posenc_tokens(const void* x, const float* pos, void* tokens, int B, int C, int H, int W, int pos_w,
                  int oy, int ox, int dtype, cudaStream_t st, const int* crop = nullptr);
int tokens_to_nchw(const void* tokens, void* out, int B, int C, int H, int W, int dtype, cudaStream_t st);
int zone_masks(const uint8_t* mask, uint8_t* zm, uint8_t* hm, uint8_t* pm, int B, int H, int W,
               const cfp_geom& g, cudaStream_t st);

// k_hist.cu
int hist_encoder(const float* hist, void* o32, void* o64, void* o128, int64_t rows, const cfp_hist_w& w,
                 int dtype, cudaStream_t st);

// k_loftr.cu
int d2i(void* feat0, const void* emb, const void* zone_tok, const float* pos2, const uint8_t* mask, int B,
        int H, int W, int C, int S, const cfp_geom& g, const cfp_loftr_w& w, int assign, char* ws,
        const WsLayout& L, int dtype, cudaStream_t st);
int dapm_attention(const void* feat0, void* msg_map, int B, int H, int W, int C, const cfp_geom& g,
                   const cfp_loftr_w& w, char* ws, const WsLayout& L, int dtype, cudaStream_t st);
int twins(void* feat0, void* out_nchw, int B, int H, int W, int C, const cfp_twins_w& w, char* ws, const WsLayout& L,
          int dtype, cudaStream_t st);     // out_nchw != nullptr: the result goes to that NCHW map instead of feat0

// k_conv.cu
// out = conv3x3(cat[in0, in1]) + shift (+ residual); in1 may be null; in1 is read as zero inside
// the rectangle (zy0..zy1, zx0..zx1).
int conv3x3(const void* in0, const void* in1, const float* w_t, const float* shift, const void* residual,
            void* out, int B, int H, int W, int C, int zy0, int zy1, int zx0, int zx1, int dtype,
            cudaStream_t st);
int sr_conv_ln(const void* feat0, float* sr_tok, int B, int H, int W, int C, int ws, const float* sr_t,
               const float* sr_b, const float* g, const float* b, int dtype, cudaStream_t st);

// k_lkpm.cu
int dwconv_bn_relu(const void* in, void* out, int B, int H, int W, int C, int ksize, const float* dw_t,
                   const float* dw_shift, int dtype, cudaStream_t st, int relu = 1);
int lkpm_mlp(void* feat0, const void* y, int64_t rows, int C, const cfp_lkpm_w& w, int dtype,
             cudaStream_t st);

// k_conv_tc.cu  (bf16, tcgen05)
int conv3x3_tc(const void* in0, const void* in1, const void* wpk, const float* shift, const void* residual, void* out,
               int B, int H, int W, int C, int zy0, int zy1, int zx0, int zx1, cudaStream_t st);

// k_chain_tc.cu  (bf16, tcgen05)
// y: dwconv output, token-major [rows][C] when planar_w == 0, else planar [frames][C][H][planar_pitch] of frames with
// planar_n = H * planar_w tokens
int lkpm_mlp_tc(void* feat0, const void* y, int64_t rows, int planar_n, int planar_w, int planar_pitch, int C, const cfp_lkpm_w& w,
                cudaStream_t st);
int sr_conv_ln_tc(const void* feat0, float* sr_tok, int B, int H, int W, int C, int ws, const void* sr_tc,
                  const float* sr_b, const float* g, const float* b, cudaStream_t st);

// k_dwconv_tc.cu  (bf16, tcgen05)
size_t dwconv_tc_plane_bytes(int B, int H, int W, int C, int K);
int dwconv_tc(const void* in, const void** planar_out, int* planar_pitch, int B, int H, int W, int C, int K, const void* toep, const float* shift,
              char* plane_ws, cudaStream_t st);

// k_train.cu  (fp32 training-step building blocks)
int tr_gemm(const float* A, int64_t a_rs, int64_t a_cs, const float* B, int64_t b_rs, int64_t b_cs, float* C, int64_t c_rs,
            int M, int N, int K, const float* bias, int accumulate, cudaStream_t st);
int tr_colsum(const float* x, float* out, int64_t rows, int C, cudaStream_t st);
int tr_bn_stats(const float* x, int64_t rows, int C, float eps, float momentum, float* mean, float* rstd, float* running_mean,
                float* running_var, float* scratch, cudaStream_t st);
int tr_bn_apply(const float* x, const float* mean, const float* rstd, const float* gamma, const float* beta, float* y,
                int64_t rows, int C, int relu, cudaStream_t st);
int tr_bn_bwd(const float* dy, const float* x, const float* mean, const float* rstd, const float* gamma, const float* beta,
              float* dx, float* dgamma, float* dbeta, int64_t rows, int C, int relu, cudaStream_t st);
int tr_ln_fwd(const float* x, const float* g, const float* b, float* y, int64_t rows, int C, float eps, cudaStream_t st);
int tr_ln_bwd(const float* x, const float* g, const float* dy, float* dx, float* dg, float* db, int64_t rows, int C, float eps,
              cudaStream_t st);
int tr_ew(const float* a, const float* b, float* out, int64_t n, int op, cudaStream_t st);
// k_train_attn.cu  (row regrouping + linear-attention building blocks of the training step)
int tr_gather_rows(const float* src, const int* idx, float* out, int64_t n, int C, cudaStream_t st);
int tr_scatter_add_rows(const float* src, const int* idx, const float* base, float* out, int64_t n, int64_t base_rows, int C,
                        cudaStream_t st);
int tr_attn_reduce(const float* A, const float* Bm, const float* w, float* KV, float* As, int G, int R, int C, int nh,
                   cudaStream_t st);
int tr_attn_apply(const float* X, const float* KV, float* out, int G, int R, int C, int nh, int transpose, cudaStream_t st);
int tr_head_dot(const float* a, const float* b, float* out, int64_t rows, int C, int nh, int rpg, float eps, cudaStream_t st);
int tr_rowop(const float* a, const float* s, const float* b, float* out, int64_t rows, int C, int nh, int rpg, int op,
             cudaStream_t st);
int tr_sumsq(const float* x, int64_t n, float scale, float* out, cudaStream_t st);
int tr_adamw(float* p, const float* g, float* m, float* v, int64_t n, const int64_t* seg_end, const float* seg_lr, int nseg,
             float beta1, float beta2, float eps, float wd, int step, float grad_scale, const float* sumsq, float max_norm,
             cudaStream_t st);
int tr_dwconv_wgrad(const float* x, const float* dy, float* dw, int B, int H, int W, int C, int K, cudaStream_t st);

// k_io.cu  (input side f3, loss / metrics f4)
int zone_hist(const float* dep, int B, int H, int W, int sy, int sx, int ph, int pw, int zn, int nbins, float max_distance,
              const double* centres, float* fh, uint8_t* mask, int* hist_out, cudaStream_t st);
int zone_samples(const float* fh, const uint8_t* mask, float* out, int64_t zones, int S, const float* w0, const float* w1, int mode,
                 cudaStream_t st);
int silog_fwd(const float* pred, const float* target, const uint8_t* mask, int B, int h, int w, int H, int W, int interpolate,
              double* scratch, float* loss, cudaStream_t st);
int silog_bwd(const float* pred, const float* target, const uint8_t* mask, int B, int h, int w, int H, int W, int interpolate,
              const double* scratch, float gout, float* grad_pred, cudaStream_t st);
int depth_metrics(const float* gt, const float* pred, const uint8_t* valid, int64_t n, double* scratch, double* out, cudaStream_t st);

// k_dec_tc.cu  (decoder shell f1, adaptive-bins head f2; bf16, channels-last)
int conv_gen_tc(const void* in, int cin, int kc, int taps, const void* wpk, const float* shift, float slope, void* out, int out_pitch,
                int out_coff, int B, int H, int W, int cout, cudaStream_t st);
int upsample_concat(const void* lo, int h, int w, int c_lo, int lo_pitch, const float* skip, int c_skip, void* out, int B, int H, int W,
                    int c_out, cudaStream_t st);
int copy_channels(const void* src, int src_pitch, void* dst, int dst_pitch, int coff, int C, int64_t rows, cudaStream_t st);
int posenc_tokens_nhwc(const void* x, int x_pitch, const float* pos, void* tokens, int B, int C, int H, int W, int pos_w, int oy, int ox,
                       cudaStream_t st);
int channel_mean(const void* x, int pitch, int C, int B, int npix, float* mean, cudaStream_t st);
int head_regressor(const float* mean, const float* wc, const float* w0, const float* b0, const float* w2, const float* b2, const float* w4,
                   const float* b4, int B, int E, int Hd, int nb, float min_val, float max_val, float* edges, float* centres,
                   cudaStream_t st);
int head_expect_tc(const void* x, int pitch, int B, int npix, const void* w_tc, const float* bias, const float* centres, int nb, float* pred,
                   float* prob, cudaStream_t st);

// k_dec_f32.cu  (decoder shell f1, adaptive-bins head f2; exact fp32 engine, channels-last)
int conv_f32(const float* in, int cin, int taps, const float* w, const float* shift, float slope, float* out, int out_pitch, int out_coff,
             int B, int H, int W, int cout, cudaStream_t st);
int upsample_concat_f32(const float* lo, int h, int w, int c_lo, int lo_pitch, const float* skip, int c_skip, float* out, int B, int H, int W,
                        int c_out, cudaStream_t st);
int copy_channels_f32(const float* src, int src_pitch, float* dst, int dst_pitch, int coff, int C, int64_t rows, cudaStream_t st);
int posenc_tokens_nhwc_f32(const float* x, int x_pitch, const float* pos, float* tokens, int B, int C, int H, int W, int pos_w, int oy, int ox,
                           cudaStream_t st);
int channel_mean_f32(const float* x, int pitch, int C, int B, int npix, float* mean, cudaStream_t st);
int head_expect_f32(const float* x, int pitch, int B, int npix, const float* w_t, const float* bias, const float* centres, int nb, float* pred,
                    float* prob, cudaStream_t st);

// k_selftest.cu
int umma_selftest(const void* A, const void* B, float* D, int rows_a, int N, int K, int row_shift, cudaStream_t st);

}  // namespace cfp
