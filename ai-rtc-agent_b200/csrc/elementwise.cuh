// HBM/latency-bound helper kernels of the per-frame path (SIMT; no tensor-core reshaping).
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace b2 {

// GroupNorm (+ optional SiLU) over NHWC fp16. The logical input is the channel concatenation of up
// to two tensors (torch.cat([h, skip], 1) of the UNet up blocks is never materialised).
struct GroupNormArgs {
    const __half* xa; int ca; int lda;
    const __half* xb; int cb; int ldb;   // xb may be null (cb = 0)
    const float* gamma; const float* beta;  // [ca+cb]
    __half* y; int ldy;                  // [nb*hw][ldy]
    int nb, hw, groups;
    float eps;
    int silu;
    float* partial;   // workspace: groupnorm_partial_floats(nb, groups) floats (per-chunk group sums)
    int* counters;    // 2*nb zero-initialised ints (grid barrier of the single-launch variant); null = two launches
};
// two launches: coalesced per-chunk statistics, then normalise (+SiLU); both fill the whole GPU
int groupnorm_launch(const GroupNormArgs& a, cudaStream_t s);
size_t groupnorm_partial_floats(int nb, int groups);
// host-only: which kernel groupnorm_launch would use.  Returns the cluster size (1/2/4/8) and fills threads per CTA and
// pixels per CTA for gn_cluster_kernel, or 0 when the whole-grid kernel is used.
int groupnorm_plan(const GroupNormArgs& a, int* threads, int* pixels_per_cta);
int groupnorm_last_launch_count();  // 1 (cooperative single launch) or 2, for the most recent call on this thread

// LayerNorm over the last dim of [rows][c] fp16 (eps 1e-5, affine), one warp per row.
int layernorm_launch(const __half* x, int ldx, const float* gamma, const float* beta, __half* y, int ldy,
                     long rows, int c, float eps, cudaStream_t s);

// nearest-neighbour x2 upsample NHWC fp16 (Upsample2D / nn.Upsample before the 3x3 conv)
int upsample2x_launch(const __half* x, __half* y, int nb, int h, int w, int c, cudaStream_t s);

// Direct 3x3 conv (pad 1, stride 1) for tiny Cin (<= 4): UNet conv_in (4->320), TAESD encoder head
// (3->64, reads the u8 NHWC video frame and applies 1/255), TAESD decoder head (4->64, tanh(z/3)*3 in,
// ReLU out).  w: fp16 [cout][cin][3][3] (PyTorch OIHW), bias fp32 [cout] or null.
enum : int { SC_IN_U8 = 1, SC_IN_TANH3 = 2, SC_OUT_RELU = 4, SC_IN_F32_NCHW = 8, SC_IN_F16_NCHW = 16 };
struct SmallConvArgs {
    const void* x;       // fp16 NHWC [nb,h,w,cin] or u8 NHWC when SC_IN_U8
    const float* wt;     // fp32 [cin*9][cout], k = tap*cin + c (smallconv_prep_launch)
    const float* bias;
    __half* y; int ldy;  // NHWC [nb,h,w,cout]
    int nb, h, w_, cin, cout;
    int in_h, in_w;      // source extents (nearest resize when != h,w; VaeImageProcessor.resize)
    int flags;
    int uc_rows;         // batch rows n < uc_rows read source row n, rows n >= uc_rows read row n - uc_rows:
                         // the source is cat(x[0:uc_rows], x) (UNet input of classifier-free guidance); 0 = identity
};
int smallconv_launch(const SmallConvArgs& a, cudaStream_t s);
// OIHW fp16 -> fp32 [cin*9][cout] (once, at load time)
int smallconv_prep_launch(const __half* w_oihw, float* wt, int cout, int cin, cudaStream_t s);

// StreamDiffusion scheduler_step_batch + stream-batch buffer update (predict_x0_batch), fused.
//   x0[i] = c_out[i] * (x[i] - beta[i]*eps[i]) / alpha[i] + c_skip[i] * x[i]
//   out_latent = x0[T-1];  x[i+1] = alpha[i+1]*x0[i] + beta[i+1]*noise[i+1]   (i < T-1)
// x, eps: [T][hw][4] fp16; noise: [T][hw][4] fp16; coef: fp32 [4][T] = alpha, beta, c_skip, c_out.
int lcm_step_launch(__half* x, const __half* eps, const __half* noise, const float* coef, __half* out_latent,
                    int T, int hw, int do_add_noise, cudaStream_t s);

// The same with StreamDiffusion's classifier-free guidance (unet_step, guidance_scale > 1), one launch.  cfg_type is
// B2SD_CFG_SELF / _INITIALIZE / _FULL; eps holds the UNet batch, uncond rows first: 0 (self), 1 (initialize) or T (full) of
// them, then the T text rows.  stock: stock_noise [T][hw][4] fp16, read and updated in place.  Per slot i:
//   s = stock after the T > 1 shift cat(noise[0:1], stock[:-1]); initialize: s[0] = eps[0]
//   eps_uncond = full ? eps[i] : delta * s[i];  pred = eps_uncond + guidance * (eps_text[i] - eps_uncond)
//   x0[i] = scheduler_step(pred, x[i]);  buffer update and out_latent as lcm_step
//   self / initialize: stock[i] = noise[(i+1) % T] + scheduler_step(pred, beta[i] s[i]) * alpha[i+1] / beta[i+1]
//   (alpha[T] = beta[T] = 1); full: stock[i] = s[i]
enum : int { CFG_NONE = 0, CFG_SELF = 1, CFG_INITIALIZE = 2, CFG_FULL = 3 };
int lcm_cfg_step_launch(__half* x, const __half* eps, const __half* noise, __half* stock, const float* coef, __half* out_latent,
                        int T, int hw, int do_add_noise, int cfg_type, float guidance, float delta, cudaStream_t s);

// Decoder tail + lib/pipeline.py:72-74 + image_utils.postprocess_image, on the fp16 grid:
//   y16 (decoder conv out, fp16) -> y*2-1 -> /2+0.5 -> clamp(0,1) -> *255 -> clamp -> trunc to u8, NCHW
int post_u8_launch(const __half* y_nhwc, int ldy, uint8_t* out_nchw, int nb, int h, int w, cudaStream_t s);
// StreamDiffusion.__call__ return value: fp16 NCHW image = y*2-1 (DecoderTiny tail), roughly [-1,1]
int post_f16_launch(const __half* y_nhwc, int ldy, __half* out_nchw, int nb, int h, int w, cudaStream_t s);

// fp32 tiny linear for prepare-time work: out[b][n] = bias[n] + sum_k act(in[b][k]) * W[n][k]
int small_linear_launch(const float* in, int in_ld, const __half* w, const float* bias, float* out, int out_ld,
                        int nb, int n, int k, int silu_in, cudaStream_t s);
// sinusoidal timestep embedding [cos | sin], fp32 [nb][dim]
int timestep_embedding_launch(const float* t, float* out, int nb, int dim, cudaStream_t s);

// dtype / layout helpers used when weights are loaded
int cast_f32_to_f16_launch(const float* x, __half* y, long n, cudaStream_t s);
int cast_f16_to_f32_launch(const __half* x, float* y, long n, cudaStream_t s);
// OIHW (fp16) -> packed [O][dst_ld] at column offset koff, K order [tap][c] for channels [c0, c0+cn)
int pack_conv_weight_launch(const __half* w_oihw, __half* dst, int dst_ld, int koff, int o, int i, int taps,
                            int c0, int cn, cudaStream_t s);
// copy rows with a row permutation: dst[r][:] = src[perm[r]][:]
int gather_rows_launch(const __half* src, int src_ld, const int* perm, __half* dst, int dst_ld, int rows, int cols,
                       cudaStream_t s);

// LayerNorm folded into its consumer GEMM, load-time preparation on packed [rows][k] fp16 weights:
//   scale_cols: W'[n][k] = W[n][k] * gamma[k];  row_sum: s[n] = sum_k W'[n][k];  row_dot: b'[n] = sum_k W[n][k] * beta[k] (+ bias[n])
int scale_cols_launch(__half* w, long rows, int k, const float* gamma, cudaStream_t s);
int row_sum_launch(const __half* w, long rows, int k, float* out, cudaStream_t s);
int row_dot_launch(const __half* w, long rows, int k, const float* v, const float* bias, float* out, cudaStream_t s);

}  // namespace b2
