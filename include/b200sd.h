/*
 * libb200sd -- C ABI of the B200-native per-frame img2img path.
 *
 * The reference (yondonfu/ai-rtc-agent) has no C/FFI boundary of its own: its drop-in boundary is
 * two Python classes (lib/pipeline.py:17-96 StreamDiffusionPipeline, lib/wrapper.py:34-407
 * StreamDiffusionWrapper) that reach the GPU through TensorRT engines built by the un-vendored
 * `streamdiffusion` package.  This header is what the Python shim in
 * ai-rtc-agent_b200/host/ binds with ctypes (see INTEGRATION.md); every entry point names the
 * reference call it stands in for.
 *
 * Conventions: plain pointers and sizes only (no torch types); all device pointers are CUDA device
 * memory of the current device; `stream` is a cudaStream_t passed as void*; every function returns 0
 * on success and non-zero on failure, with the message available from b2sd_last_error().
 * No function synchronises the device unless its comment says so.
 */
#ifndef B200SD_H
#define B200SD_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

const char* b2sd_last_error(void);
int b2sd_version(void);

/* ------------------------------------------------------------------------------------------------
 * Operator level (the contractions inside the reference's unet.engine / vae_*.engine,
 * lib/wrapper.py:445-466): used by the parity tests and by the engine below.
 * ---------------------------------------------------------------------------------------------- */

/* NHWC fp16 view: element (n,h,w,c) at ptr[((n*H + h)*W + w)*ld + c] */
typedef struct {
    const void* ptr;
    int n, h, w, c;
    int ld;
} b2sd_act_view;

enum {
    B2SD_IG_RELU = 1,
    B2SD_IG_GEGLU = 2,
    B2SD_IG_TCONV = 64,      /* run the persistent halo-tile kernel (stride-1 3x3, 64 -> 64 channels: the TAESD body) */
    B2SD_IG_PAIR = 128       /* CTA pairs: tcgen05.mma.cta_group::2 (M = 256 per MMA), each CTA stages half of the weight tile;
                                normal orientation, bn % 32 == 0, splits <= 4 */
};

/* conv3x3 / conv1x1 / Linear as one implicit GEMM:
 *   out[row][j] = acc_scale * (sum_seg sum_tap sum_c src[seg](row, tap, c) * w[j][k] + colbias[b][j])
 *                 + res_scale * res[row][j]        (then ReLU / GEGLU per flags)
 * K order of the packed weight rows = segments in sequence, each [tap][c]. */
typedef struct {
    b2sd_act_view src[3];
    int ntap[3];       /* 1 or 9 (3x3, pad 1) */
    int nseg;
    const void* w;     /* fp16 [w_rows][w_ld] */
    int w_rows, w_ld;
    int stride;        /* 1 or 2 */
    int nb, ho, wo;    /* output extents */
    int bn;            /* N tile, 0 = auto */
    int splits;        /* split-K factor (1, 2, 4 or 8 K slices reduced inside a thread-block cluster), <=1 = off */
    void* partial;     /* no workspace is needed (cluster split-K); optional int64 [ctas][8] debug timeline, else NULL */
    void* out;         /* fp16 [nb*ho*wo][ldc] */
    int ldc;
    const float* colbias;
    int colbias_bstride;
    const void* res;   /* fp16, indexed like out with pitch ldr */
    int ldr;
    float acc_scale, res_scale;
    int flags;
    int n_valid;       /* output channels */
    int swap;          /* 1: swapped orientation (output channels on the MMA M side, bn = 64/128/256 pixels on N) */
    /* LayerNorm without a LayerNorm launch (BasicTransformerBlock norm1/2/3), all optional (NULL / 0 = off):
     * rowstat_out  producer: also accumulate (sum, sum of squares) of every stored fp16 output row as 2^20 fixed point into
     *              uint64 [rows][2] with integer atomics (order independent => bit reproducible); caller zeroes it;
     * rowstat_in   consumer: those statistics for this GEMM's A rows; with colsum[n] = sum_k w[n][k] (w = W diag(gamma)) and
     *              colbias[n] = sum_k W[n][k] beta[k] + b[n] the epilogue computes rstd*(acc - mean*colsum) + colbias,
     *              i.e. LayerNorm(A) W^T + b, mean/var over ln_c columns with eps ln_eps;
     * out2         columns >= col2 are stored transposed, out2[(col - col2)*ld2 + row] (V^T block of a fused q/k/v projection). */
    void* rowstat_out;
    const void* rowstat_in;
    const float* colsum;
    int ln_c;
    float ln_eps;
    void* out2;
    int ld2, col2;
} b2sd_igemm_desc;

int b2sd_op_igemm(const b2sd_igemm_desc* d, void* stream);

/* Host-only planning (no GPU, no driver call): what b2sd_op_igemm (autotile = 0: the descriptor's bn / splits / swap / flags as
 * given) or the engine's tile policy (autotile = 1: latency policy of a single frame in flight; 2: throughput policy of >= 4
 * frames in flight; allow_swap = the contraction may use the swapped orientation) would launch for this contraction.  Pointers in the descriptor only need plausible alignment.  For tests of the host logic. */
typedef struct {
    int mode;          /* 0 = igemm_kernel, 1 = igemm_pair_kernel (CTA pairs); the halo-tile kernel is requested with B2SD_IG_TCONV */
    int swap, bn, splits;
    int grid_x, grid_y, grid_z;
    int num_stages;    /* operand ring depth */
    int acc_bufs;      /* 2 = persistent over M tiles (double-buffered TMEM accumulator) */
    int total_kb, kb_per_split;   /* K in 64-channel blocks, per cluster rank */
    int tmem_cols;
    int m_tiles;       /* 128-row output tiles */
    int64_t smem_bytes, rows_total;
} b2sd_igemm_plan_info;
int b2sd_igemm_plan_dry(const b2sd_igemm_desc* d, int autotile, int allow_swap, b2sd_igemm_plan_info* out);

/* Host-only: launch shape of GroupNorm over [ca | cb] channels, hw pixels per image: cluster = CTAs per (image, group) of the
 * cluster kernel (0 = whole-grid cooperative kernel), threads per CTA, pixels per CTA. */
int b2sd_groupnorm_plan_dry(int ca, int cb, int groups, int hw, int* cluster, int* threads, int* pixels_per_cta);
uint64_t b2sd_igemm_partial_floats(int splits, int64_t rows_total, int n_valid);   /* legacy sizing helper, unused by the cluster split-K */

/* Flash attention (self / cross) of BasicTransformerBlock.attn1 / attn2 (inside unet.engine).
 * q: [nb*sq][ldq], head h at columns [h*dp, (h+1)*dp); k likewise (batch b at row b*k_bstride, 0 = shared);
 * vt = V^T: [heads*dp][ldvt] with the key index contiguous (batch b at column b*vt_bstride);
 * out: [nb*sq][ldo], head h at columns [h*d_real, (h+1)*d_real). softmax scale = d_real^-0.5. */
typedef struct {
    const void* q; int ldq;
    const void* k; int ldk; int64_t k_bstride; int64_t k_rows;
    const void* vt; int ldvt; int64_t vt_bstride; int64_t vt_cols;
    void* out; int ldo;
    int nb, heads, sq, skv, d_real, dp;
} b2sd_attn_desc;
int b2sd_op_attention(const b2sd_attn_desc* d, void* stream);

/* GroupNorm(+SiLU) over the channel concatenation [xa | xb] (xb may be NULL), NHWC fp16. */
int b2sd_op_groupnorm(const void* xa, int ca, int lda, const void* xb, int cb, int ldb, const float* gamma,
                      const float* beta, void* y, int ldy, int nb, int hw, int groups, float eps, int silu,
                      void* stream);
int b2sd_op_layernorm(const void* x, int ldx, const float* gamma, const float* beta, void* y, int ldy,
                      int64_t rows, int c, float eps, void* stream);
int b2sd_op_upsample2x(const void* x, void* y, int nb, int h, int w, int c, void* stream);
/* direct 3x3 conv for Cin in {3,4}; flags: 1 = input is u8 NHWC scaled by 1/255 (lib/pipeline.py:61),
 * 2 = tanh(x/3)*3 on the input (DecoderTiny), 4 = ReLU on the output */
int b2sd_op_smallconv(const void* x, const void* w_oihw, const float* bias, void* y, int ldy, int nb, int h,
                      int w, int cin, int cout, int in_h, int in_w, int flags, void* stream);
/* StreamDiffusion scheduler_step_batch + stream-batch buffer update (see elementwise.cuh) */
int b2sd_op_lcm_step(void* x, const void* eps, const void* noise, const float* coef, void* out_latent, int T,
                     int hw, int do_add_noise, void* stream);
/* Classifier-free guidance types of StreamDiffusion (cfg_type "none" / "self" / "initialize" / "full") */
enum { B2SD_CFG_NONE = 0, B2SD_CFG_SELF = 1, B2SD_CFG_INITIALIZE = 2, B2SD_CFG_FULL = 3 };
/* The same step with residual / full classifier-free guidance (StreamDiffusion.unet_step with guidance_scale > 1), fused:
 * eps = UNet output rows, unconditional rows first (0 for self, 1 for initialize, T for full, then T text rows);
 * stock_noise fp16 [T][hw][4] is read and updated in place.  cfg_type is B2SD_CFG_SELF / _INITIALIZE / _FULL
 * (see elementwise.cuh for the arithmetic). */
int b2sd_op_lcm_cfg_step(void* x, const void* eps, const void* noise, void* stock_noise, const float* coef, void* out_latent,
                         int T, int hw, int do_add_noise, int cfg_type, float guidance_scale, float delta, void* stream);
/* Codec boundary (SURVEY.md 8f-1; the reference's aiortc fork decodes with NVDEC / encodes with NVENC, requirements.txt:12-13,
 * and exchanges RGB tensors in HBM with lib/pipeline.py:50-51,83,96).  NV12 surface (Y plane + interleaved UV plane, pitches in
 * bytes) <-> the frame formats of b2sd_step: u8 NHWC RGB in, u8 NCHW RGB out.  flags: 0 = BT.709 limited range,
 * B2SD_CSC_BT601, B2SD_CSC_FULL_RANGE.  b2sd_codec_probe: bit 0 = libnvcuvid loadable, bit 1 = libnvidia-encode loadable. */
enum { B2SD_CSC_BT601 = 1, B2SD_CSC_FULL_RANGE = 2 };
int b2sd_op_nv12_to_rgb(const void* y, int y_pitch, const void* uv, int uv_pitch, void* rgb_nhwc, int h, int w, int flags, void* stream);
int b2sd_op_rgb_to_nv12(const void* rgb_nchw, void* y, int y_pitch, void* uv, int uv_pitch, int h, int w, int flags, void* stream);
int b2sd_codec_probe(void);
/* decoder tail + lib/pipeline.py:72-74 on the fp16 grid -> u8 NCHW */
int b2sd_op_post_u8(const void* y_nhwc, int ldy, void* out_nchw_u8, int nb, int h, int w, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Engine level: one handle == one temporal stream (one StreamDiffusion instance, lib/wrapper.py:168).
 * Replaces StreamDiffusion + UNet2DConditionModelEngine + AutoencoderKLEngine
 * (lib/wrapper.py:445-466, 494-504) for mode="img2img", use_denoising_batch=True, frame_buffer_size=1,
 * cfg_type "none" / "self" / "initialize" / "full" (b2sd_set_guidance; lib/pipeline.py:23-42 builds "self" with guidance 0).
 * ---------------------------------------------------------------------------------------------- */
typedef struct b2sd_engine* b2sd_handle;

typedef struct {
    int block_out_channels[4];   /* (320,640,1280,1280) */
    int heads[4];                /* SD-1.5: 8,8,8,8   SD-Turbo: 5,10,20,20 */
    int down_attn[4];            /* 1,1,1,0 */
    int cross_attention_dim;     /* 768 | 1024 */
    int layers_per_block;        /* 2 */
    int norm_groups;             /* 32 */
    int ctx_tokens;              /* 77 */
    int batch;                   /* len(t_index_list) * frame_buffer_size (lib/wrapper.py:159-163) */
    int height, width;           /* image size, multiples of 64 */
    int do_add_noise;            /* lib/wrapper.py:53 */
    int use_cuda_graph;          /* replay the frame program as one CUDA graph */
} b2sd_config;

int b2sd_create(const b2sd_config* cfg, b2sd_handle* out);
int b2sd_destroy(b2sd_handle h);
/* A "lane": a second engine over the SAME parameters as `parent` (one copy of the weights in HBM), with its own activations,
 * stream state and CUDA graph, so that several frames can be in flight on different CUDA streams.  cfg = NULL copies the
 * parent's; otherwise only batch / height / width may differ.  Prepare it like any engine (after the parent's first
 * b2sd_prepare, which lays the weights out).  With a 1-step stream batch (SD-Turbo) consecutive frames of ONE video stream are
 * independent, so alternating them over two lanes overlaps frame n+1 with frame n and yields bit-identical output; lanes are
 * also how several independent video streams share one GPU.  (The reference serialises everything behind a per-frame
 * torch.cuda.synchronize(), SURVEY.md 8 a-10.) */
int b2sd_create_lane(b2sd_handle parent, const b2sd_config* cfg, b2sd_handle* out);

/* Weights under diffusers state-dict names: UNet keys as-is ("down_blocks.0.resnets.0.conv1.weight"),
 * TAESD keys prefixed "vae." ("vae.encoder.layers.0.weight").  ptr may be host or device memory.
 * dtype: 0 = fp16, 1 = fp32.  Replaces the ONNX export + TensorRT build of lib/wrapper.py:785-910.
 * After the first b2sd_prepare the raw copies of parameters that only feed the packing kernels are released (set
 * B2_KEEP_RAW=1 to keep them); loading further tensors into such an engine is an error. */
int b2sd_load_tensor(b2sd_handle h, const char* key, const void* ptr, int dtype, const int64_t* shape, int ndim);

/* Packed-weight blob: the kernel-native layouts b2sd_prepare derives from the parameters (reordered convolution
 * matrices, per-head q/k/v gathers, GEGLU interleave, fused bias vectors), written once and loaded instead of
 * b2sd_load_tensor + repacking.  Replaces the reference's cached TensorRT engine files `engines--<model>/...engine`
 * (lib/wrapper.py:593-597, 896-910; build.py:11-32).  The blob depends on the architecture and the (LoRA-fused)
 * parameter values only -- not on batch, image size or prompt.  Export after b2sd_prepare; import into a fresh engine
 * (same b2sd_config architecture fields) before b2sd_prepare.  Host synchronous. */
int b2sd_export_packed(b2sd_handle h, const char* path);
int b2sd_import_packed(b2sd_handle h, const char* path);

/* StreamDiffusion.prepare (via lib/wrapper.py:197-234): fixes per-slot scalars and noise, zeroes the
 * stream-batch latent buffer, builds the frame program.  All pointers are HOST memory:
 *   prompt_embeds  fp16 [ctx_tokens][cross_attention_dim]   (CLIP output, encoded by the caller)
 *   timesteps      fp32 [batch]                             (sub_timesteps_tensor)
 *   coef           fp32 [4][batch] = alpha_prod_t_sqrt, beta_prod_t_sqrt, c_skip, c_out
 *   init_noise     fp16 [batch][4][h/8][w/8]                (NCHW, as torch.randn produced it)
 * Synchronises `stream`. */
int b2sd_prepare(b2sd_handle h, const void* prompt_embeds, const float* timesteps, const float* coef,
                 const void* init_noise, void* stream);
/* Classifier-free guidance of StreamDiffusion.prepare (guidance_scale, delta, cfg_type, negative_prompt).  Takes effect at the
 * next b2sd_prepare, like b2sd_set_concurrency.  Guidance is active when cfg_type != B2SD_CFG_NONE and guidance_scale > 1;
 * otherwise the frame program is the unguided one.  Active guidance runs the UNet on B_u rows: T (self), T + 1 (initialize:
 * [uncond slot 0 | T text rows]) or 2T (full: [T uncond | T text]), and keeps stock_noise [T][h/8][w/8][4] in the stream
 * state (zeroed by b2sd_prepare, shared by b2sd_share_stream_state, tap "stock_noise").  uncond_embeds: HOST fp16
 * [ctx_tokens][cross_attention_dim], the encoded negative prompt; required for initialize / full, may be NULL otherwise.
 * B_u must not exceed 16. */
int b2sd_set_guidance(b2sd_handle h, int cfg_type, float guidance_scale, float delta, const void* uncond_embeds);
/* StreamDiffusion.update_prompt (lib/pipeline.py:44-45): refresh the per-layer cross-attention K/V cache.  Replaces the
 * conditional prompt only; the unconditional rows of a guided batch keep the negative prompt of b2sd_set_guidance. */
int b2sd_set_prompt_embeds(b2sd_handle h, const void* prompt_embeds, void* stream);
/* lib/wrapper.py:389-407 update_t_index_list: only sub_timesteps change (alpha/beta/c_skip/c_out keep the
 * values given to b2sd_prepare -- reference behaviour).  timesteps: fp32 [batch]; the engine repeats them for the extra
 * unconditional rows of a guided UNet batch. */
int b2sd_set_timesteps(b2sd_handle h, const float* timesteps, void* stream);

/* One StreamDiffusionPipeline.__call__ (lib/pipeline.py:76-96, NVENC branch): frame_in = device u8 NHWC
 * [in_h][in_w][3] (nearest-resized to height x width if different, SURVEY a-4), frame_out = device u8 NCHW
 * [3][height][width].  Enqueues on `stream`; no host synchronisation. */
int b2sd_step(b2sd_handle h, const void* frame_in, int in_h, int in_w, void* frame_out, void* stream);

/* Same, for the reference's split call path preprocess -> predict -> postprocess (lib/pipeline.py:50-74):
 * input may be the (3,H,W) float tensor lib/pipeline.py:65 produces; output may be the fp16 NCHW image
 * in [-1,1] that StreamDiffusion.__call__ returns (lib/wrapper.py:330). */
enum { B2SD_IN_U8_NHWC = 0, B2SD_IN_F32_NCHW = 1, B2SD_IN_F16_NCHW = 2 };
enum { B2SD_OUT_U8_NCHW = 0, B2SD_OUT_F16_NCHW = 1 };
int b2sd_step_ex(b2sd_handle h, const void* frame_in, int in_kind, int in_h, int in_w, void* frame_out,
                 int out_kind, void* stream);

/* Parity/debug taps: copies a named intermediate of the last step to host memory as fp16 NHWC.
 * Names: "x_t", "unet_in", "eps" (all B_u UNet rows), "x0", "image", "conv_in", "down.I.J", "mid", "up.I.J", "stock_noise".
 * Returns the element count via *count (pass dst = NULL to query).  Synchronises `stream`. */
int b2sd_get_tensor(b2sd_handle h, const char* name, void* dst, int64_t capacity, int64_t* count, int* dims4,
                    void* stream);
/* Profiling aid: eager replay of one frame with a CUDA event after every launch, averaged over `iters`;
 * writes a JSON array [{"name","ms"},...] to json_buf.  Synchronises. */
int b2sd_profile(b2sd_handle h, const void* frame_in, int in_h, int in_w, void* frame_out, int iters,
                 char* json_buf, int64_t cap, void* stream);
/* Device time of one launch class ("igemm", "attn", "groupnorm", "layernorm", ...) of the frame program, measured by
 * replaying a CUDA graph that holds only those launches (same order, buffers and weight streaming as the frame graph).
 * ms_per_replay = average over `iters` replays; launches / flops (optional) = launches and algorithmic FLOPs per replay. */
int b2sd_profile_kind(b2sd_handle h, const char* kind, int iters, double* ms_per_replay, int* launches, double* flops,
                      void* stream);
/* number of kernel launches (graph nodes) in one b2sd_step */
/* Concurrent use of b2sd_profile_kind (one host thread and CUDA stream per lane): after b2sd_profile_gate(n) the next n calls
 * wait for each other between their warm-up and their timed replays, so the timed regions overlap.  0 / 1 switches it off. */
int b2sd_profile_gate(int participants);
int b2sd_launches_per_step(b2sd_handle h);
/* Stage pipelining of ONE stateful stream (stream batch T > 1, where frame n+1 needs frame n's latent buffer and lanes cannot
 * simply alternate): `lane` shares `owner`'s stream-batch state; the frame program of each is cut into TAESD encoder body |
 * last encoder conv + UNet + scheduler step | TAESD decoder, and only the middle stage is serialised between the lanes (one
 * CUDA event), so the encoder of frame n+1 and the decoder of frame n-1 overlap the UNet of frame n.  Both engines must be
 * lanes of one weight store with equal batch / size; call before b2sd_prepare; submit frames alternately, in order. */
int b2sd_share_stream_state(b2sd_handle lane, b2sd_handle owner);
/* How many frames will be in flight on this GPU (lanes / independent streams).  1 (default): launch policy tuned for the
 * latency of a single frame; > 1: policy tuned for throughput (smaller operand rings so CTAs of different frames share an
 * SM; from 4 frames in flight on, contractions are launched as CTA pairs -- tcgen05.mma.cta_group::2 -- without split-K: least
 * SM time per contraction).
 * Takes effect at the next b2sd_prepare. */
int b2sd_set_concurrency(b2sd_handle h, int frames_in_flight);

#ifdef __cplusplus
}
#endif
#endif /* B200SD_H */
