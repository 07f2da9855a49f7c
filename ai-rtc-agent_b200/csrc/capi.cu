// extern "C" surface of libb200sd.so (declared in include/b200sd.h).
#include "../../include/b200sd.h"

#include "attention.cuh"
#include "codec.cuh"
#include "elementwise.cuh"
#include "igemm.cuh"
#include "tconv.cuh"

using namespace b2;

extern "C" {

const char* b2sd_last_error(void) { return b2_last_error(); }
int b2sd_version(void) { return 1; }

static ActView to_view(const b2sd_act_view& v) {
    ActView a;
    a.ptr = reinterpret_cast<const __half*>(v.ptr);
    a.N = v.n; a.H = v.h; a.W = v.w; a.C = v.c; a.ld = v.ld;
    return a;
}

static void to_igemm_desc(const b2sd_igemm_desc* d, IgemmDesc& g) {
    g.nseg = d->nseg;
    for (int s = 0; s < d->nseg && s < IG_MAX_SRC; ++s) {
        g.src[s] = to_view(d->src[s]);
        g.ntap[s] = d->ntap[s];
    }
    g.w = reinterpret_cast<const __half*>(d->w);
    g.w_rows = d->w_rows;
    g.w_ld = d->w_ld;
    g.stride = d->stride;
    g.Nb = d->nb; g.Ho = d->ho; g.Wo = d->wo;
    g.BN = d->bn;
    g.swap = d->swap;
    g.pair = (d->flags & B2SD_IG_PAIR) ? 1 : 0;
    g.splits = d->splits;
    g.partial = nullptr;
    g.dbg_ts = reinterpret_cast<unsigned long long*>(d->partial);  // op-level entry: `partial` doubles as the debug timeline buffer
    g.epi.out = reinterpret_cast<__half*>(d->out);
    g.epi.ldc = d->ldc;
    g.epi.colbias = d->colbias;
    g.epi.colbias_bstride = d->colbias_bstride;
    g.epi.res = reinterpret_cast<const __half*>(d->res);
    g.epi.ldr = d->ldr;
    g.epi.acc_scale = d->acc_scale;
    g.epi.res_scale = d->res_scale;
    g.epi.flags = d->flags & (IG_RELU | IG_GEGLU);
    g.epi.n_valid = d->n_valid;
    g.epi.rowstat_out = static_cast<unsigned long long*>(d->rowstat_out);
    g.epi.rowstat_in = static_cast<const unsigned long long*>(d->rowstat_in);
    g.epi.colsum = d->colsum;
    g.epi.ln_inv_c = d->ln_c > 0 ? 1.f / (float)d->ln_c : 0.f;
    g.epi.ln_eps = d->ln_eps;
    g.epi.out2 = reinterpret_cast<__half*>(d->out2);
    g.epi.ld2 = d->ld2;
    g.epi.col2 = d->col2;
}

int b2sd_op_igemm(const b2sd_igemm_desc* d, void* stream) {
    if (!d) {
        b2_set_error("b2sd_op_igemm: null desc");
        return -1;
    }
    IgemmDesc g{};
    to_igemm_desc(d, g);
    if (d->flags & B2SD_IG_TCONV) {   // the persistent halo-tile kernel (64 -> 64 channel 3x3 convolutions)
        TconvPlan tp;
        if (tconv_plan(g, &tp)) return -1;
        return tconv_launch(tp, reinterpret_cast<cudaStream_t>(stream));
    }
    IgemmPlan plan;
    if (igemm_plan(g, &plan)) return -1;
    return igemm_launch(plan, reinterpret_cast<cudaStream_t>(stream));
}

int b2sd_igemm_plan_dry(const b2sd_igemm_desc* d, int autotile, int allow_swap, b2sd_igemm_plan_info* out) {
    if (!d || !out) {
        b2_set_error("b2sd_igemm_plan_dry: null argument");
        return -1;
    }
    IgemmDesc g{};
    to_igemm_desc(d, g);
    g.dbg_ts = nullptr;
    IgemmPlan plan;
    if (autotile == 2) {   // the engine's throughput policy (b2sd_set_concurrency >= 4): 100 KB rings, CTA pairs without split-K
        g.ring_kb = 100; g.max_splits = 4; g.pair_auto = 1; g.pair_splits = 1;
    }
    igemm_set_dry_run(true);
    const int rc = autotile ? igemm_autotile(g, allow_swap != 0, &plan) : igemm_plan(g, &plan);
    igemm_set_dry_run(false);
    if (rc) return -1;
    out->mode = plan.mode;
    out->swap = plan.p.swap;
    out->bn = plan.p.BN;
    out->splits = plan.splits;
    out->grid_x = (int)plan.grid.x; out->grid_y = (int)plan.grid.y; out->grid_z = (int)plan.grid.z;
    out->num_stages = plan.p.num_stages;
    out->acc_bufs = plan.p.acc_bufs;
    out->total_kb = plan.p.total_kb;
    out->kb_per_split = plan.p.kb_per_split;
    out->tmem_cols = (int)plan.p.tmem_cols;
    out->m_tiles = plan.p.tiles_w * plan.p.tiles_h * plan.p.tiles_n;
    out->smem_bytes = (int64_t)plan.smem;
    out->rows_total = plan.rows_total;
    return 0;
}

int b2sd_groupnorm_plan_dry(int ca, int cb, int groups, int hw, int* cluster, int* threads, int* pixels_per_cta) {
    GroupNormArgs a{};
    a.ca = ca; a.cb = cb; a.lda = ca; a.ldb = cb; a.ldy = ca + cb; a.groups = groups; a.hw = hw; a.nb = 1;
    if (groups <= 0 || hw <= 0 || ca <= 0 || !cluster) {
        b2_set_error("b2sd_groupnorm_plan_dry: bad arguments");
        return -1;
    }
    *cluster = groupnorm_plan(a, threads, pixels_per_cta);
    return 0;
}

uint64_t b2sd_igemm_partial_floats(int splits, int64_t rows_total, int n_valid) {
    return igemm_partial_floats(splits, rows_total, n_valid);
}

int b2sd_op_nv12_to_rgb(const void* y, int y_pitch, const void* uv, int uv_pitch, void* rgb_nhwc, int h, int w, int flags, void* stream) {
    return nv12_to_rgb_u8_launch(static_cast<const uint8_t*>(y), y_pitch, static_cast<const uint8_t*>(uv), uv_pitch,
                                 static_cast<uint8_t*>(rgb_nhwc), h, w, flags, reinterpret_cast<cudaStream_t>(stream));
}
int b2sd_op_rgb_to_nv12(const void* rgb_nchw, void* y, int y_pitch, void* uv, int uv_pitch, int h, int w, int flags, void* stream) {
    return rgb_u8_to_nv12_launch(static_cast<const uint8_t*>(rgb_nchw), static_cast<uint8_t*>(y), y_pitch, static_cast<uint8_t*>(uv),
                                 uv_pitch, h, w, flags, reinterpret_cast<cudaStream_t>(stream));
}
int b2sd_codec_probe(void) { return codec_probe(); }

int b2sd_op_attention(const b2sd_attn_desc* d, void* stream) {
    AttnDesc a{};
    a.q = reinterpret_cast<const __half*>(d->q); a.ldq = d->ldq;
    a.k = reinterpret_cast<const __half*>(d->k); a.ldk = d->ldk; a.k_bstride = d->k_bstride; a.k_rows = d->k_rows;
    a.vt = reinterpret_cast<const __half*>(d->vt); a.ldvt = d->ldvt; a.vt_bstride = d->vt_bstride; a.vt_cols = d->vt_cols;
    a.out = reinterpret_cast<__half*>(d->out); a.ldo = d->ldo;
    a.nb = d->nb; a.heads = d->heads; a.sq = d->sq; a.skv = d->skv; a.d_real = d->d_real; a.dp = d->dp;
    AttnPlan plan;
    if (attn_plan(a, &plan)) return -1;
    return attn_launch(plan, reinterpret_cast<cudaStream_t>(stream));
}

int b2sd_op_groupnorm(const void* xa, int ca, int lda, const void* xb, int cb, int ldb, const float* gamma,
                      const float* beta, void* y, int ldy, int nb, int hw, int groups, float eps, int silu,
                      void* stream) {
    GroupNormArgs a{};
    a.xa = reinterpret_cast<const __half*>(xa); a.ca = ca; a.lda = lda;
    a.xb = reinterpret_cast<const __half*>(xb); a.cb = cb; a.ldb = ldb;
    a.gamma = gamma; a.beta = beta;
    a.y = reinterpret_cast<__half*>(y); a.ldy = ldy;
    a.nb = nb; a.hw = hw; a.groups = groups; a.eps = eps; a.silu = silu;
    static float* scratch = nullptr;   // op-level entry only (tests); the engine passes its own workspace
    static size_t scratch_floats = 0;
    const size_t need = groupnorm_partial_floats(nb, groups);
    if (need > scratch_floats) {
        if (scratch) cudaFree(scratch);
        if (cudaMalloc(&scratch, need * sizeof(float)) != cudaSuccess) {
            b2_set_error("b2sd_op_groupnorm: cudaMalloc failed");
            return -1;
        }
        scratch_floats = need;
    }
    a.partial = scratch;
    static int* gn_counters = nullptr;
    if (!gn_counters) {
        if (cudaMalloc(&gn_counters, 64 * sizeof(int)) != cudaSuccess || cudaMemset(gn_counters, 0, 64 * sizeof(int)) != cudaSuccess) {
            b2_set_error("b2sd_op_groupnorm: counter alloc failed");
            return -1;
        }
    }
    a.counters = gn_counters;
    return groupnorm_launch(a, reinterpret_cast<cudaStream_t>(stream));
}

int b2sd_op_layernorm(const void* x, int ldx, const float* gamma, const float* beta, void* y, int ldy,
                      int64_t rows, int c, float eps, void* stream) {
    return layernorm_launch(reinterpret_cast<const __half*>(x), ldx, gamma, beta, reinterpret_cast<__half*>(y), ldy,
                            rows, c, eps, reinterpret_cast<cudaStream_t>(stream));
}

int b2sd_op_upsample2x(const void* x, void* y, int nb, int h, int w, int c, void* stream) {
    return upsample2x_launch(reinterpret_cast<const __half*>(x), reinterpret_cast<__half*>(y), nb, h, w, c,
                             reinterpret_cast<cudaStream_t>(stream));
}

int b2sd_op_smallconv(const void* x, const void* w_oihw, const float* bias, void* y, int ldy, int nb, int h,
                      int w, int cin, int cout, int in_h, int in_w, int flags, void* stream) {
    SmallConvArgs a{};
    static float* wt = nullptr;  // op-level entry only: re-prepared on every call
    if (!wt && cudaMalloc(&wt, 36 * 1024 * sizeof(float)) != cudaSuccess) {
        b2_set_error("b2sd_op_smallconv: cudaMalloc failed");
        return -1;
    }
    if (cout > 1024 || smallconv_prep_launch(reinterpret_cast<const __half*>(w_oihw), wt, cout, cin, reinterpret_cast<cudaStream_t>(stream)))
        return -1;
    a.x = x; a.wt = wt; a.bias = bias;
    a.y = reinterpret_cast<__half*>(y); a.ldy = ldy;
    a.nb = nb; a.h = h; a.w_ = w; a.cin = cin; a.cout = cout; a.in_h = in_h; a.in_w = in_w; a.flags = flags;
    return smallconv_launch(a, reinterpret_cast<cudaStream_t>(stream));
}

int b2sd_op_lcm_step(void* x, const void* eps, const void* noise, const float* coef, void* out_latent, int T,
                     int hw, int do_add_noise, void* stream) {
    return lcm_step_launch(reinterpret_cast<__half*>(x), reinterpret_cast<const __half*>(eps),
                           reinterpret_cast<const __half*>(noise), coef, reinterpret_cast<__half*>(out_latent), T, hw,
                           do_add_noise, reinterpret_cast<cudaStream_t>(stream));
}

int b2sd_op_lcm_cfg_step(void* x, const void* eps, const void* noise, void* stock_noise, const float* coef, void* out_latent,
                         int T, int hw, int do_add_noise, int cfg_type, float guidance_scale, float delta, void* stream) {
    return lcm_cfg_step_launch(reinterpret_cast<__half*>(x), reinterpret_cast<const __half*>(eps),
                               reinterpret_cast<const __half*>(noise), reinterpret_cast<__half*>(stock_noise), coef,
                               reinterpret_cast<__half*>(out_latent), T, hw, do_add_noise, cfg_type, guidance_scale, delta,
                               reinterpret_cast<cudaStream_t>(stream));
}

int b2sd_op_post_u8(const void* y_nhwc, int ldy, void* out_nchw_u8, int nb, int h, int w, void* stream) {
    return post_u8_launch(reinterpret_cast<const __half*>(y_nhwc), ldy, reinterpret_cast<uint8_t*>(out_nchw_u8), nb,
                          h, w, reinterpret_cast<cudaStream_t>(stream));
}

}  // extern "C"
