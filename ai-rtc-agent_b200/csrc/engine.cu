// Per-frame engine: TAESD encoder -> stream-batched UNet -> LCM step -> TAESD decoder, assembled once
// (at b2sd_prepare) as a static list of kernel launches over preallocated HBM buffers and replayed as
// a CUDA graph.  Mirrors what the reference reaches through StreamDiffusion.__call__
// (lib/wrapper.py:330) and its three TensorRT engines (lib/wrapper.py:445-466).
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <atomic>
#include <chrono>
#include <functional>
#include <thread>
#include <map>
#include <memory>
#include <string>
#include <vector>

#include "../../include/b200sd.h"
#include "attention.cuh"
#include "elementwise.cuh"
#include "igemm.cuh"
#include "tconv.cuh"

using namespace b2;

#define CUDA_OK(expr)                                                                       \
    do {                                                                                    \
        cudaError_t e__ = (expr);                                                           \
        if (e__ != cudaSuccess) {                                                           \
            b2_set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), __FILE__, __LINE__); \
            return -1;                                                                      \
        }                                                                                   \
    } while (0)
#define TRY(expr)            \
    do {                     \
        if ((expr) != 0) return -1; \
    } while (0)

namespace {

struct Act {
    __half* p = nullptr;
    int n = 0, h = 0, w = 0, c = 0, ld = 0;
    long elems() const { return (long)n * h * w * ld; }
};

struct Raw {  // a loaded parameter, fp16 on device (+ host fp32 copy for 1-D tensors)
    __half* p = nullptr;      // null once released (pack-only parameters after the first successful prepare)
    bool pack_only = false;   // only ever read by the packing kernels (3x3 / shortcut convs, q/k/v, GEGLU, Cin<=4 convs)
    std::vector<int64_t> shape;
    std::vector<float> host;
    long numel() const {
        long v = 1;
        for (auto s : shape) v *= s;
        return v;
    }
};

// bump allocator over cudaMalloc'ed slabs (HBM is plentiful: no reuse, no fragmentation)
class Arena {
  public:
    explicit Arena(size_t slab) : slab_(slab) {}
    ~Arena() { release(); }
    void* alloc(size_t bytes) {
        bytes = (bytes + 1023) & ~size_t(1023);
        if (cur_ < 0 || off_ + bytes > sizes_[cur_]) {
            // find next slab that fits, else allocate
            int next = cur_ + 1;
            while (next < (int)slabs_.size() && sizes_[next] < bytes) ++next;
            if (next >= (int)slabs_.size()) {
                size_t sz = bytes > slab_ ? bytes : slab_;
                void* p = nullptr;
                if (cudaMalloc(&p, sz) != cudaSuccess) return nullptr;
                slabs_.push_back(p);
                sizes_.push_back(sz);
                next = (int)slabs_.size() - 1;
            }
            cur_ = next;
            off_ = 0;
        }
        void* r = static_cast<char*>(slabs_[cur_]) + off_;
        off_ += bytes;
        return r;
    }
    void reset() { cur_ = slabs_.empty() ? -1 : 0; off_ = 0; }
    void release() {
        for (void* p : slabs_) cudaFree(p);
        slabs_.clear();
        sizes_.clear();
        cur_ = -1;
        off_ = 0;
    }

  private:
    size_t slab_;
    std::vector<void*> slabs_;
    std::vector<size_t> sizes_;
    int cur_ = -1;
    size_t off_ = 0;
};

struct Op {
    std::function<int(cudaStream_t)> fn;
    std::string name;
    double flops = 0.0;  // algorithmic 2*MAC count of the launch (0 for non-contraction kernels)
    template <class F>
    Op(F f, std::string n = "", double fl = 0.0) : fn(std::move(f)), name(std::move(n)), flops(fl) {}
    int operator()(cudaStream_t s) const { return fn(s); }
};

}  // namespace

// ------------------------------------------------------------------------------------------------
// Tile / split-K policy of the frame program (batch-1 driven; derived from the cold-weight sweep in
// profiles/r01_tile_sweep.md, not from a model).  Fills `plan` for the chosen (BN, splits, orientation).
// allow_swap: the caller is a UNet contraction (never TAESD / V^T / GEGLU).  Host-only: works in igemm dry-run mode.
static int igemm_autotile_single(IgemmDesc d, bool allow_swap, IgemmPlan* plan_out);

// Tile policy + CTA pairs.  The single-CTA policy picks orientation, N tile and split-K.  With d.pair_auto (set by the engine
// when several frames are in flight) a normal-orientation result with >= 2 M tiles and an N tile that is a multiple of 32 is
// re-planned as CTA pairs (igemm_pair_kernel) with the same N tile and the split-K factor capped at d.pair_splits: under
// concurrency the GPU is filled by the other frames, so what counts is SM time per contraction, and a pair stages half the
// weight bytes per SM, has a deeper ring in the same shared memory and needs no cluster reduction (same-box A/B, 6 lanes:
// 440.6 -> 470.5 frames/s; the same tiles WITHOUT pairing: 433.0; pairs with the latency policy's split-K: 417.6;
// profiles/ab_r02u.txt, ab_r02x.txt).  Tuning overrides: B2_PAIR=0/1/2, B2_PAIR_SPLITS=n, B2_PAIR_SINGLE=1 (control: re-plan
// with the capped split-K but single CTAs).
int igemm_autotile(IgemmDesc d, bool allow_swap, IgemmPlan* plan_out) {
    TRY(igemm_autotile_single(d, allow_swap, plan_out));
    static const char* pair_env = getenv("B2_PAIR");
    static const char* ps_env = getenv("B2_PAIR_SPLITS");
    static const bool pair_single = getenv("B2_PAIR_SINGLE") != nullptr;
    const int pair_mode = pair_env ? atoi(pair_env) : d.pair_auto;
    const int pair_splits = ps_env ? atoi(ps_env) : (d.pair_splits > 0 ? d.pair_splits : 4);
    const IgemmPlan& pl = *plan_out;
    const int m_tiles = pl.p.tiles_w * pl.p.tiles_h * pl.p.tiles_n;
    if (pair_mode <= 0 || pl.p.swap || m_tiles < 2 || (pl.p.BN % 32) != 0) return 0;
    if (pair_mode == 2 && pl.p.total_kb < 20) return 0;
    d.swap = 0; d.BN = pl.p.BN; d.splits = pl.splits > pair_splits ? pair_splits : pl.splits; d.partial = nullptr;
    d.pair = pair_single ? 0 : 1;
    IgemmPlan paired;
    if (igemm_plan(d, &paired)) return 0;   // keep the single-CTA plan
    *plan_out = paired;
    return 0;
}

static int igemm_autotile_single(IgemmDesc d, bool allow_swap, IgemmPlan* plan_out) {
    IgemmPlan& plan = *plan_out;
    const bool geglu = (d.epi.flags & IG_GEGLU) != 0;
    const int n_gemm = geglu ? 2 * d.epi.n_valid : d.epi.n_valid;
    static const bool swap_on = getenv("B2_SWAP") != nullptr, swap_off = getenv("B2_NO_SWAP") != nullptr;
    static const bool tuned = getenv("B2_NO_TUNED_TILES") == nullptr;
    static const char* ms_env = getenv("B2_MAX_SPLITS");   // tuning: cap of the cluster split-K factor (throughput vs latency)
    const int max_splits = ms_env ? atoi(ms_env) : (d.max_splits > 0 ? d.max_splits : 8);
    int total_kb = 0;
    for (int sidx = 0; sidx < d.nseg && sidx < IG_MAX_SRC; ++sidx) total_kb += d.ntap[sidx] * (d.src[sidx].C / IG_BK);
    const long rows_all = (long)d.Nb * d.Ho * d.Wo;
    // Swapped orientation by default only where it measured faster (tools/bench_op.py, cold weights): the 8x8 level,
    // where a 128-pixel M tile would be half empty.  B2_SWAP=1 forces it for every eligible UNet contraction.
    const bool swap_here = allow_swap && !geglu && d.epi.n_valid >= 128 && (d.epi.n_valid & 7) == 0 &&
                           (swap_on || (!swap_off && tuned && rows_all <= 64 && total_kb >= 90));
    if (swap_here) {
        d.swap = 1;
        d.BN = rows_all >= 256 ? 256 : (rows_all >= 128 ? 128 : 64);
        d.splits = 1; d.partial = nullptr;
        TRY(igemm_plan(d, &plan));
        const long ctas = (long)plan.grid.x * plan.grid.y;
        int max_by_k = plan.p.total_kb / 4;
        if (max_by_k < 1) max_by_k = 1;
        if (max_by_k > 8) max_by_k = 8;
        int splits = 1;
        while (splits * 2 <= max_by_k && ctas * splits * 2 <= 192 && splits * 2 <= max_splits) splits *= 2;
        if (splits > 1) {
            d.splits = splits;
            TRY(igemm_plan(d, &plan));
        }
        return 0;
    }
    d.swap = 0;
    auto vt_ok = [&](int bn) { return !d.epi.out2 || d.epi.col2 % bn == 0; };   // fused q/k/v: an N tile is all q/k or all v
    if (tuned && !geglu && n_gemm % 160 == 0 && total_kb >= 40 && vt_ok(160)) {
        // K-heavy contractions that cannot fill the GPU with 160-wide tiles alone (batch 1): wide tiles + cluster
        // split-K beat 64-wide tiles (profiles/r01_tile_sweep.md: -10..-40 % per launch, weights streamed from HBM)
        d.BN = 160; d.splits = 1; d.partial = nullptr;
        TRY(igemm_plan(d, &plan));
        const int m_tiles = plan.p.tiles_w * plan.p.tiles_h * plan.p.tiles_n;
        const long tiles = (long)m_tiles * (n_gemm / 160);
        int bn = 0, splits = 0;
        if (tiles < 132) {
            if (m_tiles >= 8) { bn = 160; splits = 4; }
            else if (m_tiles >= 2 && n_gemm % 256 == 0 && total_kb >= 180 && vt_ok(256)) { bn = 256; splits = 8; }
        }
        if (bn && splits > max_splits) bn = 0;   // capped: fall through to the generic choice below
        if (bn) {
            d.BN = bn; d.splits = splits;
            TRY(igemm_plan(d, &plan));
            return 0;
        }
    }
    static const int cands[] = {256, 160, 128, 64, 32, 16};
    std::vector<int> valid;
    for (int bn : cands) {
        if (geglu && (bn % 32 != 0 || bn < 64)) continue;
        if (n_gemm % bn == 0 && vt_ok(bn)) valid.push_back(bn);
    }
    if (valid.empty()) {  // ragged N: one masked tile size
        int bn = 16;
        while (bn < n_gemm && bn < 128) bn <<= 1;
        valid.push_back(bn);
    }
    for (int bn : valid) {
        if (bn < 64 && n_gemm >= 64) break;  // narrow tiles re-read A too often: prefer split-K below
        d.BN = bn; d.splits = 1; d.partial = nullptr;
        TRY(igemm_plan(d, &plan));
        if ((long)plan.grid.x * plan.grid.y >= 132) return 0;
    }
    // not enough tiles for one wave: smallest reasonable tile, then split K
    int bn = valid.back();
    for (int v : valid) if (v >= 64) bn = v;  // smallest >= 64 if any (valid is descending)
    d.BN = bn; d.splits = 1; d.partial = nullptr;
    TRY(igemm_plan(d, &plan));
    const long ctas = (long)plan.grid.x * plan.grid.y;
    int splits = ctas >= 96 ? 1 : (int)((148 + ctas - 1) / ctas);
    if (tuned && ctas >= 64 && total_kb <= 12) splits = 1;   // the cluster reduction (~3 us) costs more than 5 k-blocks
    const int max_by_k = plan.p.total_kb / 4 > 0 ? plan.p.total_kb / 4 : 1;
    if (splits > max_by_k) splits = max_by_k;
    if (splits > 8) splits = 8;
    while (splits > max_splits && splits > 1) splits >>= 1;
    if (geglu) splits = 1;
    if (splits > 1) {
        d.splits = splits;
        TRY(igemm_plan(d, &plan));
    }
    return 0;
}

// Parameters and everything derived from them (kernel-native packed layouts, fused fp32 vectors).  Read-only on the frame
// path, so several engines ("lanes", b2sd_create_lane) share one store: one copy of the 1.7 GB UNet in HBM however many
// frames are in flight.
struct WeightStore {
    std::map<std::string, Raw> raw;
    Arena weights{256u << 20};   // packed parameters + the raw ones kernels read directly (live for the store's lifetime)
    Arena raw_only{256u << 20};  // raw parameters that only feed the packing kernels: released after the first prepare
    bool raw_released = false;
    bool imported = false;       // parameters came from a packed blob (b2sd_import_packed)
    std::map<std::string, __half*> packed;   // cache of packed weight matrices
    std::map<std::string, float*> fvec;      // cache of fp32 vectors
    std::map<std::string, size_t> packed_bytes, fvec_bytes;   // their sizes (b2sd_export_packed)
};

struct b2sd_engine {
    b2sd_config cfg{};
    int lh = 0, lw = 0;  // latent extents
    std::shared_ptr<WeightStore> ws;
    std::map<std::string, Raw>& raw;
    Arena& weights;
    Arena& raw_only;
    bool& raw_released;
    bool& imported;
    std::map<std::string, __half*>& packed;
    std::map<std::string, float*>& fvec;
    std::map<std::string, size_t>& packed_bytes;
    std::map<std::string, size_t>& fvec_bytes;
    Arena state{16u << 20};      // stream state + small persistent vectors
    Arena prog{512u << 20};      // activations / per-program buffers (reset at prepare)
    explicit b2sd_engine(std::shared_ptr<WeightStore> s)
        : ws(std::move(s)), raw(ws->raw), weights(ws->weights), raw_only(ws->raw_only), raw_released(ws->raw_released),
          imported(ws->imported), packed(ws->packed), fvec(ws->fvec), packed_bytes(ws->packed_bytes), fvec_bytes(ws->fvec_bytes) {}

    // persistent stream state (StreamDiffusion attributes)
    Act x_in;             // UNet input batch: slot 0 = fresh x_t, slots 1.. = x_t_latent_buffer
    __half* noise = nullptr;   // init_noise, NHWC [B][lh][lw][4]
    float* coef = nullptr;     // [4][B]
    float* tsteps = nullptr;   // [B]
    __half* ctx = nullptr;     // prompt embeddings [ctx_tokens][D]
    float* temb_sin = nullptr; // [B][C0]
    float* temb_h = nullptr;   // [B][4*C0]
    float* temb = nullptr;     // [B][4*C0]
    float* gn_ws = nullptr;    // GroupNorm chunk partials (shared: launches are stream-ordered)
    int* tile_counters = nullptr;
    float coef_host[4][64]{};
    // classifier-free guidance (b2sd_set_guidance): requested settings, and the ones the current program was built with
    struct Guidance { int cfg_type = B2SD_CFG_NONE; float scale = 1.f, delta = 1.f; };
    Guidance guide_req, guide;     // guide.cfg_type == NONE unless guidance is active (cfg_type != none and scale > 1)
    std::vector<__half> uncond_host;
    int uc_rows = 0;               // unconditional rows in front of the T text rows of the UNet batch: 0, 1 (initialize), T (full)
    int rows_cap = 0;              // UNet rows tsteps / temb* / gn_ws are sized for
    __half* stock = nullptr;       // stock_noise NHWC [T][lh][lw][4]
    __half* uctx = nullptr;        // unconditional prompt embeddings [ctx_tokens][D]
    __half* ctx_rows = nullptr;    // guided batch with uncond rows: per-row prompt embeddings [B_u][Lpad][D] (zero padded)
    int unet_rows() const { return cfg.batch + uc_rows; }

    unsigned long long* ln_stats = nullptr;   // slab of per-row LayerNorm statistics [rows][2] (see IgEpilogue::rowstat_out)
    size_t ln_stats_cap = 0, ln_stats_used = 0;   // in 64-bit words
    std::vector<Op> prog_frame, prog_prompt, prog_time;
    std::map<std::string, Act> taps;
    SmallConvArgs head{};   // encoder head (reads the caller's frame)
    Act image;              // decoder output, fp16 NHWC (ld 8)
    bool built = false;
    int concurrency = 1;   // frames expected in flight on this GPU (b2sd_set_concurrency): > 1 selects the throughput launch policy
    int launches = 0;
    std::string cur;   // name prefix of the layer being built (debug / profiling labels)
    bool allow_swap = false;  // builders enable the swapped GEMM orientation for UNet contractions (never TAESD / V^T / GEGLU)
    cudaGraphExec_t graph_exec = nullptr;
    cudaGraph_t graph = nullptr;
    // Stage pipelining of a stateful (T > 1) stream over lanes that SHARE the stream-batch state (b2sd_share_stream_state): the
    // frame program is cut into [TAESD encoder body | last encoder conv + UNet + scheduler step | TAESD decoder], three CUDA
    // graphs; only the middle stage touches the shared x_in, and the lanes chain it through one event.
    struct StageGroup { cudaEvent_t unet_done = nullptr; ~StageGroup() { if (unet_done) cudaEventDestroy(unet_done); } };
    std::shared_ptr<StageGroup> group;
    size_t idx_enc_end = 0, idx_unet_end = 0;          // stage boundaries inside prog_frame
    cudaGraphExec_t stage_exec[3] = {nullptr, nullptr, nullptr};
    cudaGraph_t stage_graph[3] = {nullptr, nullptr, nullptr};
    void drop_graphs() {
        if (graph_exec) { cudaGraphExecDestroy(graph_exec); graph_exec = nullptr; }
        if (graph) { cudaGraphDestroy(graph); graph = nullptr; }
        for (int i = 0; i < 3; ++i) {
            if (stage_exec[i]) { cudaGraphExecDestroy(stage_exec[i]); stage_exec[i] = nullptr; }
            if (stage_graph[i]) { cudaGraphDestroy(stage_graph[i]); stage_graph[i] = nullptr; }
        }
    }

    ~b2sd_engine() { drop_graphs(); }

    // ---- parameters -----------------------------------------------------------------------------
    const Raw* get(const std::string& key) {
        auto it = raw.find(key);
        if (it == raw.end()) {
            b2_set_error("missing weight '%s'", key.c_str());
            return nullptr;
        }
        return &it->second;
    }
    bool has(const std::string& key) const { return raw.count(key) != 0; }

    // fp32 device vector = sum of the named 1-D parameters (optionally row-permuted)
    float* vec(const std::vector<std::string>& keys, const std::vector<int>* perm = nullptr, int pad_to = 0) {
        std::string ck = "v:";
        for (auto& k : keys) ck += k + "+";
        if (perm) ck += "perm";
        auto it = fvec.find(ck);
        if (it != fvec.end()) return it->second;
        std::vector<float> host;
        for (auto& k : keys) {
            const Raw* r = get(k);
            if (!r) return nullptr;
            if (host.empty()) host.assign(r->host.begin(), r->host.end());
            else
                for (size_t i = 0; i < host.size() && i < r->host.size(); ++i) host[i] += r->host[i];
        }
        if (perm) {
            std::vector<float> t(perm->size());
            for (size_t i = 0; i < perm->size(); ++i) t[i] = (*perm)[i] >= 0 ? host[(*perm)[i]] : 0.f;
            host.swap(t);
        }
        if ((int)host.size() < pad_to) host.resize(pad_to, 0.f);
        float* d = static_cast<float*>(weights.alloc(host.size() * sizeof(float)));
        if (!d) return nullptr;
        if (cudaMemcpy(d, host.data(), host.size() * sizeof(float), cudaMemcpyHostToDevice) != cudaSuccess) return nullptr;
        fvec[ck] = d;
        fvec_bytes[ck] = host.size() * sizeof(float);
        return d;
    }

    // fp32 [cin*9][cout] weights of a tiny-Cin conv (cached)
    const float* small_w(const std::string& key, cudaStream_t s) {
        auto it = fvec.find("sw:" + key);
        if (it != fvec.end()) return it->second;
        const Raw* r = get(key);
        if (!r) return nullptr;
        if (!r->p) { b2_set_error("parameter '%s' was released after the first prepare and is not in the packed cache", key.c_str()); return nullptr; }
        const int cout = (int)r->shape[0], cin = (int)r->shape[1];
        float* d = static_cast<float*>(weights.alloc((size_t)cin * 9 * cout * sizeof(float)));
        if (!d || smallconv_prep_launch(r->p, d, cout, cin, s)) return nullptr;
        fvec["sw:" + key] = d;
        fvec_bytes["sw:" + key] = (size_t)cin * 9 * cout * sizeof(float);
        return d;
    }

    struct ConvSeg { std::string key; int c0, cn, taps; };
    // packed [rows_pad][K] matrix, K = concat of segments each ordered [tap][c]
    __half* pack_conv(const std::string& name, const std::vector<ConvSeg>& segs, int rows, int* k_out,
                      cudaStream_t s) {
        int K = 0;
        for (auto& g : segs) K += g.taps * g.cn;
        *k_out = K;
        auto it = packed.find(name);
        if (it != packed.end()) return it->second;
        const int rows_pad = (rows + 15) / 16 * 16;
        __half* dst = static_cast<__half*>(weights.alloc((size_t)rows_pad * K * 2));
        if (!dst) return nullptr;
        cudaMemsetAsync(dst, 0, (size_t)rows_pad * K * 2, s);
        int koff = 0;
        for (auto& g : segs) {
            const Raw* r = get(g.key);
            if (!r) return nullptr;
            if (!r->p) { b2_set_error("parameter '%s' was released after the first prepare and is not in the packed cache", g.key.c_str()); return nullptr; }
            const int cin_total = (int)r->shape[1];
            if (pack_conv_weight_launch(r->p, dst, K, koff, rows, cin_total, g.taps, g.c0, g.cn, s)) return nullptr;
            koff += g.taps * g.cn;
        }
        packed[name] = dst;
        packed_bytes[name] = (size_t)rows_pad * K * 2;
        return dst;
    }
    // rows gathered from one or more [*, K] matrices: spec = list of (key, perm)
    __half* pack_rows(const std::string& name, const std::vector<std::pair<std::string, std::vector<int>>>& parts,
                      int K, cudaStream_t s) {
        auto it = packed.find(name);
        if (it != packed.end()) return it->second;
        size_t rows = 0;
        for (auto& p : parts) rows += p.second.size();
        const size_t rows_pad = (rows + 15) / 16 * 16;
        __half* dst = static_cast<__half*>(weights.alloc(rows_pad * K * 2));
        if (!dst) return nullptr;
        cudaMemsetAsync(dst, 0, rows_pad * K * 2, s);
        size_t r0 = 0;
        for (auto& p : parts) {
            const Raw* r = get(p.first);
            if (!r) return nullptr;
            if (!r->p) { b2_set_error("parameter '%s' was released after the first prepare and is not in the packed cache", p.first.c_str()); return nullptr; }
            int* dperm = static_cast<int*>(weights.alloc(p.second.size() * sizeof(int)));
            if (!dperm) return nullptr;
            cudaMemcpyAsync(dperm, p.second.data(), p.second.size() * sizeof(int), cudaMemcpyHostToDevice, s);
            cudaStreamSynchronize(s);  // host vector may die before the copy otherwise
            if (gather_rows_launch(r->p, K, dperm, dst + r0 * K, K, (int)p.second.size(), K, s)) return nullptr;
            r0 += p.second.size();
        }
        packed[name] = dst;
        packed_bytes[name] = rows_pad * K * 2;
        return dst;
    }

    // LayerNorm folded into a consumer GEMM (IgEpilogue::colsum): W' = gather(parts) diag(gamma) in place of the gathered rows,
    // colsum[n] = sum_k W'[n][k], bias'[n] = sum_k W[n][k] beta[k] + bias[n].  Cached like every packed parameter.
    struct LnFold { __half* w = nullptr; const float* colsum = nullptr; const float* bias = nullptr; };
    int fold_ln(const std::string& name, const std::vector<std::pair<std::string, std::vector<int>>>& parts, int K,
                const std::string& ln_prefix, const float* bias_vec, LnFold* out, cudaStream_t s) {
        size_t rows = 0;
        for (auto& p : parts) rows += p.second.size();
        const size_t rows_pad = (rows + 15) / 16 * 16;
        const bool done = packed.count(name) && fvec.count(name + ":cs") && fvec.count(name + ":b");
        __half* w = pack_rows(name, parts, K, s);
        if (!w) return -1;
        if (!done) {
            const float* gamma = vec({ln_prefix + ".weight"});
            const float* beta = vec({ln_prefix + ".bias"});
            float* cs = static_cast<float*>(weights.alloc(rows_pad * sizeof(float)));
            float* bb = static_cast<float*>(weights.alloc(rows_pad * sizeof(float)));
            if (!gamma || !beta || !cs || !bb) return -1;
            cudaMemsetAsync(bb, 0, rows_pad * sizeof(float), s);
            TRY(row_dot_launch(w, (long)rows, K, beta, bias_vec, bb, s));     // on the un-scaled rows
            TRY(scale_cols_launch(w, (long)rows_pad, K, gamma, s));
            TRY(row_sum_launch(w, (long)rows_pad, K, cs, s));
            fvec[name + ":cs"] = cs; fvec_bytes[name + ":cs"] = rows_pad * sizeof(float);
            fvec[name + ":b"] = bb; fvec_bytes[name + ":b"] = rows_pad * sizeof(float);
        }
        out->w = w;
        out->colsum = fvec[name + ":cs"];
        out->bias = fvec[name + ":b"];
        return 0;
    }
    unsigned long long* alloc_rowstat(long rows) {
        if (ln_stats_used + 2 * (size_t)rows > ln_stats_cap) {
            b2_set_error("LayerNorm statistics slab exhausted");
            return nullptr;
        }
        unsigned long long* p = ln_stats + ln_stats_used;
        ln_stats_used += 2 * (size_t)rows;
        return p;
    }

    // ---- program construction helpers -----------------------------------------------------------
    Act new_act(int n, int h, int w, int c, int ld = 0) {
        Act a;
        a.n = n; a.h = h; a.w = w; a.c = c; a.ld = ld ? ld : c;
        a.p = static_cast<__half*>(prog.alloc((size_t)a.elems() * 2));
        return a;
    }
    static ActView view(const Act& a) { return ActView{a.p, a.n, a.h, a.w, a.c, a.ld}; }
    static ActView tokens(const Act& a) { return ActView{a.p, 1, 1, a.n * a.h * a.w, a.c, a.ld}; }

    // choose N tile / split-K for a good grid (igemm_autotile), plan, and append the launch
    // append a planned contraction
    void push_igemm(std::vector<Op>& dst, const IgemmPlan& plan, const std::string& label, double flops) {
        if (&dst == &prog_frame) launches += 1;
        dst.push_back(Op([plan](cudaStream_t s) { return igemm_launch(plan, s); }, label, flops));
    }

    // choose N tile / split-K for a good grid (igemm_autotile), plan, and append the launch
    int add_igemm(std::vector<Op>& dst, IgemmDesc d) {
        const bool geglu = (d.epi.flags & IG_GEGLU) != 0;
        const int n_gemm = geglu ? 2 * d.epi.n_valid : d.epi.n_valid;
        const bool extras = d.epi.rowstat_out || d.epi.colsum || d.epi.out2;   // not implemented by the swapped-orientation epilogue
        // several frames in flight: a 100 KB operand ring lets CTAs of different frames share an SM (measured +5.5 % throughput
        // at 3 lanes; one frame alone prefers the 200 KB ring on launches with <= 1 CTA per SM)
        if (concurrency > 1 && d.ring_kb == 0) d.ring_kb = 100;
        // ... and spreading one contraction over fewer K slices costs latency but less SM time (cluster reduction): +1.5 %
        if (concurrency > 1 && d.max_splits == 0) d.max_splits = 4;
        // ... and with the GPU filled by >= 4 frames, CTA pairs without split-K use the least SM time per contraction
        // (igemm_autotile): +6.8 % at 6 lanes, +11 % at 8.  Two stage-pipelined lanes of ONE stateful stream (T > 1) run mostly
        // one UNet at a time and keep split-K: pairs there measured -14 % (SD-1.5 4-step 512^2, profiles/ab_sd15_r02z.txt).
        if (concurrency >= 4 && d.pair_auto == 0) { d.pair_auto = 1; d.pair_splits = 1; }
        IgemmPlan plan;
        TRY(igemm_autotile(d, allow_swap && !extras, &plan));
        if (d.epi.out2 && d.epi.col2 % plan.p.BN != 0) {   // an N tile must be all q/k or all v (igemm_autotile filters on it)
            b2_set_error("fused q/k/v projection: N tile %d does not divide the V offset %d", plan.p.BN, d.epi.col2);
            return -1;
        }
        char label[256];
        snprintf(label, sizeof(label), "igemm %s rows=%ld n=%d kb=%d bn=%d splits=%d grid=%u,%u,%u %s", cur.c_str(),
                 plan.rows_total, d.epi.n_valid, plan.p.total_kb, plan.p.BN, plan.splits, plan.grid.x, plan.grid.y,
                 plan.grid.z, plan.p.swap ? "swapped" : (plan.pair ? "pairs" : "taps"));
        push_igemm(dst, plan, label, 2.0 * (double)plan.rows_total * n_gemm * plan.p.total_kb * IG_BK);
        return 0;
    }

    int add_groupnorm(const Act& xa, const Act* xb, const std::string& prefix, const Act& y, float eps, int silu) {
        GroupNormArgs a{};
        a.xa = xa.p; a.ca = xa.c; a.lda = xa.ld;
        if (xb) { a.xb = xb->p; a.cb = xb->c; a.ldb = xb->ld; }
        a.gamma = vec({prefix + ".weight"});
        a.beta = vec({prefix + ".bias"});
        if (!a.gamma || !a.beta) return -1;
        a.y = y.p; a.ldy = y.ld;
        a.nb = xa.n; a.hw = xa.h * xa.w; a.groups = cfg.norm_groups; a.eps = eps; a.silu = silu;
        a.partial = gn_ws;
        a.counters = tile_counters;   // zero-initialised, self re-arming
        launches += 1;
        prog_frame.push_back(Op([a](cudaStream_t s) { return groupnorm_launch(a, s); }, "groupnorm " + prefix));
        return 0;
    }

    int add_layernorm(const Act& x, const std::string& prefix, const Act& y) {
        const float* g = vec({prefix + ".weight"});
        const float* b = vec({prefix + ".bias"});
        if (!g || !b) return -1;
        const long rows = (long)x.n * x.h * x.w;
        const __half* xp = x.p; __half* yp = y.p;
        const int ldx = x.ld, ldy = y.ld, c = x.c;
        ++launches;
        prog_frame.push_back(Op([=](cudaStream_t s) { return layernorm_launch(xp, ldx, g, b, yp, ldy, rows, c, 1e-5f, s); }, "layernorm " + prefix));
        return 0;
    }

    // conv3x3 (or 1x1) over one source with bias / relu / residual
    int add_conv(std::vector<Op>& dst, const Act& x, const std::string& wkey, const std::string& bkey, int taps,
                 int stride, const Act& y, int flags, const Act* res, cudaStream_t s, float acc_scale = 1.f,
                 float res_scale = 1.f) {
        const Raw* w = get(wkey);
        if (!w) return -1;
        cur = wkey;
        const int cout = (int)w->shape[0];
        int K = 0;
        __half* wp = pack_conv(wkey, {{wkey, 0, x.c, taps}}, cout, &K, s);
        if (!wp) return -1;
        IgemmDesc d{};
        d.nseg = 1; d.src[0] = view(x); d.ntap[0] = taps;
        d.w = wp; d.w_rows = (cout + 15) / 16 * 16; d.w_ld = K;
        d.stride = stride;
        d.Nb = y.n; d.Ho = y.h; d.Wo = y.w;
        d.epi.out = y.p; d.epi.ldc = y.ld;
        if (!bkey.empty()) {
            d.epi.colbias = vec({bkey}, nullptr, 16);
            if (!d.epi.colbias) return -1;
        }
        d.epi.colbias_bstride = 0;
        if (res) { d.epi.res = res->p; d.epi.ldr = res->ld; }
        d.epi.acc_scale = acc_scale; d.epi.res_scale = res_scale;
        d.epi.flags = flags;
        d.epi.n_valid = cout;
        // the TAESD body at 256x256 and above: persistent halo-tile kernel with resident weights (tconv.cu)
        static const bool no_tconv = getenv("B2_NO_TCONV") != nullptr;
        static const char* tc_min = getenv("B2_TCONV_MIN_TILES");
        const long tiles = (long)y.n * ((y.h + TC_TH - 1) / TC_TH) * ((y.w + TC_TW - 1) / TC_TW);
        if (!no_tconv && stride == 1 && tconv_eligible(d) && tiles >= (tc_min ? atoi(tc_min) : 2 * 148)) {
            TconvPlan tp;
            TRY(tconv_plan(d, &tp));
            char label[256];
            snprintf(label, sizeof(label), "tconv %s rows=%ld tiles=%d grid=%u nbuf=%d", wkey.c_str(), tp.rows_total, tp.p.num_tiles,
                     tp.grid.x, tp.p.nbuf);
            if (&dst == &prog_frame) launches += 1;
            dst.push_back(Op([tp](cudaStream_t st) { return tconv_launch(tp, st); }, label, 2.0 * (double)tp.rows_total * cout * K));
            return 0;
        }
        return add_igemm(dst, d);
    }

    // Linear over tokens: y = x W^T (+bias) (+res)
    struct LinExtra {   // LayerNorm-fold / row-statistics / transposed-V options of a Linear (IgEpilogue)
        unsigned long long* rowstat_out = nullptr;
        const unsigned long long* rowstat_in = nullptr;
        const float* colsum = nullptr;
        int ln_c = 0;
        __half* out2 = nullptr;
        int ld2 = 0, col2 = 0;
    };
    int add_linear(std::vector<Op>& dst, const ActView& x, const __half* w, int n, int k, const float* bias,
                   __half* out, int ldc, const __half* res, int ldr, int flags = 0, int n_valid = -1,
                   const LinExtra* ex = nullptr) {
        IgemmDesc d{};
        if (ex) {
            d.epi.rowstat_out = ex->rowstat_out;
            d.epi.rowstat_in = ex->rowstat_in;
            d.epi.colsum = ex->colsum;
            d.epi.ln_inv_c = ex->ln_c ? 1.f / (float)ex->ln_c : 0.f;
            d.epi.ln_eps = 1e-5f;
            d.epi.out2 = ex->out2; d.epi.ld2 = ex->ld2; d.epi.col2 = ex->col2;
        }
        d.nseg = 1; d.src[0] = x; d.ntap[0] = 1;
        d.w = w; d.w_rows = n; d.w_ld = k;
        d.stride = 1;
        d.Nb = 1; d.Ho = 1; d.Wo = x.W;
        d.epi.out = out; d.epi.ldc = ldc;
        d.epi.colbias = bias; d.epi.colbias_bstride = 0;
        d.epi.res = res; d.epi.ldr = ldr;
        d.epi.acc_scale = 1.f; d.epi.res_scale = 1.f;
        d.epi.flags = flags;
        d.epi.n_valid = n_valid >= 0 ? n_valid : n;
        return add_igemm(dst, d);
    }

    int build_resnet(const std::string& p, const Act& xa, const Act* xb, int cout, Act* out, cudaStream_t s);
    int build_transformer(const std::string& p, const Act& x, int heads, Act* out, cudaStream_t s);
    int build_taesd_block(const std::string& p, const Act& x, Act* out, cudaStream_t s);
    int build_program(cudaStream_t s);
    int run_range(std::vector<Op>& ops, size_t a, size_t b, cudaStream_t s) {
        for (size_t i = a; i < b && i < ops.size(); ++i) TRY(ops[i](s));
        return 0;
    }
    int run(std::vector<Op>& ops, cudaStream_t s) {
        static const bool dbg = getenv("B200SD_DEBUG_SYNC") != nullptr;
        static const char* skip = getenv("B200SD_SKIP");  // debug: "groupnorm,attn" drops those launches (timing only)
        static const char* skip_name = getenv("B200SD_SKIP_NAME");  // debug: drop launches whose label contains this substring
        int idx = 0;
        for (auto& op : ops) {
            if (skip) {
                const std::string kind = op.name.substr(0, op.name.find(' '));
                if (!kind.empty() && std::string(skip).find(kind) != std::string::npos) { ++idx; continue; }
            }
            if (skip_name && op.name.find(skip_name) != std::string::npos) { ++idx; continue; }
            TRY(op(s));
            if (dbg) {
                cudaError_t e = cudaStreamSynchronize(s);
                if (e != cudaSuccess) {
                    b2_set_error("op %d '%s' failed: %s", idx, op.name.c_str(), cudaGetErrorString(e));
                    fprintf(stderr, "b2sd: op %d '%s' failed: %s\n", idx, op.name.c_str(), cudaGetErrorString(e));
                    return -1;
                }
            }
            ++idx;
        }
        return 0;
    }
};

// ------------------------------------------------------------------------------------------------
// ResnetBlock2D (diffusers resnet.py): GN+SiLU -> conv1 (+temb) -> GN+SiLU -> conv2, + shortcut(x)
int b2sd_engine::build_resnet(const std::string& p, const Act& xa, const Act* xb, int cout, Act* out, cudaStream_t s) {
    cur = p;
    allow_swap = true;
    const int cin = xa.c + (xb ? xb->c : 0);
    const int B = xa.n;
    Act n1 = new_act(B, xa.h, xa.w, cin);
    TRY(add_groupnorm(xa, xb, p + "norm1", n1, 1e-5f, 1));
    // conv1 with per-sample column bias = conv1.bias + time_emb_proj(silu(emb))
    Act h1 = new_act(B, xa.h, xa.w, cout);
    {
        int K = 0;
        __half* wp = pack_conv(p + "conv1.weight", {{p + "conv1.weight", 0, cin, 9}}, cout, &K, s);
        if (!wp) return -1;
        float* colbias = static_cast<float*>(prog.alloc((size_t)B * cout * sizeof(float)));
        const float* bsum = vec({p + "conv1.bias", p + "time_emb_proj.bias"});
        const Raw* wt = get(p + "time_emb_proj.weight");
        if (!colbias || !bsum || !wt) return -1;
        const int tdim = (int)wt->shape[1];
        const float* emb = temb;
        const __half* wtp = wt->p;
        prog_time.push_back(Op([=](cudaStream_t st) { return small_linear_launch(emb, tdim, wtp, bsum, colbias, cout, B, cout, tdim, 1, st); }, "temb " + p));
        IgemmDesc d{};
        d.nseg = 1; d.src[0] = view(n1); d.ntap[0] = 9;
        d.w = wp; d.w_rows = cout; d.w_ld = K; d.stride = 1;
        d.Nb = B; d.Ho = xa.h; d.Wo = xa.w;
        d.epi.out = h1.p; d.epi.ldc = h1.ld;
        d.epi.colbias = colbias; d.epi.colbias_bstride = cout;
        d.epi.acc_scale = 1.f; d.epi.res_scale = 1.f; d.epi.n_valid = cout;
        TRY(add_igemm(prog_frame, d));
    }
    Act n2 = new_act(B, xa.h, xa.w, cout);
    TRY(add_groupnorm(h1, nullptr, p + "norm2", n2, 1e-5f, 1));
    *out = new_act(B, xa.h, xa.w, cout);
    IgemmDesc d{};
    d.stride = 1; d.Nb = B; d.Ho = xa.h; d.Wo = xa.w;
    d.epi.out = out->p; d.epi.ldc = out->ld;
    d.epi.acc_scale = 1.f; d.epi.res_scale = 1.f; d.epi.n_valid = cout;
    d.src[0] = view(n2); d.ntap[0] = 9;
    int K = 0;
    if (has(p + "conv_shortcut.weight")) {
        // out = conv2(n2) + conv_shortcut(cat[xa, xb]): one K loop over three TMA sources
        std::vector<ConvSeg> segs = {{p + "conv2.weight", 0, cout, 9}, {p + "conv_shortcut.weight", 0, xa.c, 1}};
        d.nseg = 2; d.src[1] = view(xa); d.ntap[1] = 1;
        if (xb) {
            segs.push_back({p + "conv_shortcut.weight", xa.c, xb->c, 1});
            d.nseg = 3; d.src[2] = view(*xb); d.ntap[2] = 1;
        }
        __half* wp = pack_conv(p + "conv2+shortcut", segs, cout, &K, s);
        if (!wp) return -1;
        d.w = wp; d.w_rows = cout; d.w_ld = K;
        d.epi.colbias = vec({p + "conv2.bias", p + "conv_shortcut.bias"});
    } else {
        if (xb) {
            b2_set_error("resnet %s: concat input without conv_shortcut", p.c_str());
            return -1;
        }
        __half* wp = pack_conv(p + "conv2.weight", {{p + "conv2.weight", 0, cout, 9}}, cout, &K, s);
        if (!wp) return -1;
        d.nseg = 1;
        d.w = wp; d.w_rows = cout; d.w_ld = K;
        d.epi.colbias = vec({p + "conv2.bias"});
        d.epi.res = xa.p; d.epi.ldr = xa.ld;
    }
    if (!d.epi.colbias) return -1;
    return add_igemm(prog_frame, d);
}

// Transformer2DModel + BasicTransformerBlock (diffusers transformer_2d.py / attention.py)
int b2sd_engine::build_transformer(const std::string& p, const Act& x, int heads, Act* out, cudaStream_t s) {
    cur = p;
    allow_swap = true;
    const int B = x.n, C = x.c, HW = x.h * x.w;
    const long M = (long)B * HW;
    const int d_real = C / heads;
    const int dp = d_real <= 64 ? 64 : (d_real <= 128 ? 128 : 192);
    const int Cp = heads * dp;
    const int D = cfg.cross_attention_dim, L = cfg.ctx_tokens;
    const std::string t = p + "transformer_blocks.0.";
    auto head_perm = [&](int base) {  // packed row (h*dp+i) <- source row (h*d+i), -1 = zero padding
        std::vector<int> pm(Cp);
        for (int hh = 0; hh < heads; ++hh)
            for (int i = 0; i < dp; ++i) pm[hh * dp + i] = i < d_real ? base + hh * d_real + i : -1;
        return pm;
    };
    Act n = new_act(B, x.h, x.w, C);
    TRY(add_groupnorm(x, nullptr, p + "norm", n, 1e-6f, 0));
    const int HWp = (HW + 7) / 8 * 8;
    const bool one_gemm = (HW % 8 == 0) || B == 1;   // V^T of all batch items is one [Cp][B*HW] matrix (TMA needs 16-byte column origins)
    // LayerNorm folding + fused q/k/v projection: norm1/2/3 never run as kernels.  Each LayerNorm input is produced by a Linear
    // whose epilogue also accumulates the row statistics (rowstat_out); the consumer GEMM runs on the RAW rows with gamma folded
    // into its weights and applies mean / rstd in its epilogue (IgEpilogue::colsum).  B2_NO_LNFOLD=1 restores the three
    // layernorm launches + separate V^T GEMM (also used when the batch's V^T columns need per-image padding).
    // Measured (profiles/ab_sd15_r02l.txt, ab_r02l.txt), with the consumer's colsum / bias' vectors staged in shared memory:
    // SD-Turbo 512x512 4 lanes 380 -> 421 fps, SD-1.5 4-step 512x512 124 -> 133 fps, 768x768 50.1 -> 52.9 fps.  (A first
    // version that read those vectors from global memory inside the per-chunk loop LOST 5 % at 16384 tokens.)
    static const bool no_fold = getenv("B2_NO_LNFOLD") != nullptr;
    static const char* fold_rows_env = getenv("B2_LNFOLD_MAX_ROWS");   // tuning: disable the fold above this many tokens
    const long fold_max_rows = fold_rows_env ? atol(fold_rows_env) : (1l << 40);
    const bool fold = !no_fold && one_gemm && (long)B * (cfg.height / 8) * (cfg.width / 8) <= fold_max_rows;
    const int inner = 4 * C;
    std::vector<int> gperm;   // GEGLU: weight rows interleaved per 128-wide tile as [64 value | 64 gate]
    {
        const int half = 64;
        for (int tI = 0; tI < inner / half; ++tI) {
            for (int i = 0; i < half; ++i) gperm.push_back(tI * half + i);
            for (int i = 0; i < half; ++i) gperm.push_back(inner + tI * half + i);
        }
    }
    const float* bff1 = vec({t + "ff.net.0.proj.bias"}, &gperm);
    if (!bff1) return -1;
    // proj_in: Linear (SD-Turbo) or 1x1 conv (SD-1.5) -- the same GEMM on NHWC tokens
    const Raw* wpi = get(p + "proj_in.weight");
    if (!wpi) return -1;
    Act hs = new_act(B, x.h, x.w, C);
    unsigned long long *st1 = nullptr, *st2 = nullptr, *st3 = nullptr;
    if (fold) {
        st1 = alloc_rowstat(M); st2 = alloc_rowstat(M); st3 = alloc_rowstat(M);
        if (!st1 || !st2 || !st3) return -1;
    }
    {
        LinExtra ex; ex.rowstat_out = st1;
        TRY(add_linear(prog_frame, tokens(n), wpi->p, C, C, vec({p + "proj_in.bias"}), hs.p, C, nullptr, 0, 0, -1, &ex));
    }
    // ---- self attention
    Act qk = new_act(1, 1, (int)M, 2 * Cp);
    const long vt_ld = one_gemm ? (M + 7) / 8 * 8 : (long)B * HWp;
    const long vt_bstride = one_gemm ? HW : HWp;
    __half* vt = static_cast<__half*>(prog.alloc((size_t)Cp * vt_ld * 2));
    if (!vt) return -1;
    cudaMemsetAsync(vt, 0, (size_t)Cp * vt_ld * 2, s);  // pad columns must stay finite (0 * NaN = NaN in P.V)
    if (fold) {
        // one GEMM: [q | k | v] rows; q/k columns go to `qk`, the V block is stored transposed (K-major V^T for the P.V MMA)
        LnFold f;
        TRY(fold_ln(t + "attn1.qkv+ln", {{t + "attn1.to_q.weight", head_perm(0)}, {t + "attn1.to_k.weight", head_perm(0)},
                                         {t + "attn1.to_v.weight", head_perm(0)}}, C, t + "norm1", nullptr, &f, s));
        LinExtra ex; ex.rowstat_in = st1; ex.colsum = f.colsum; ex.ln_c = C; ex.out2 = vt; ex.ld2 = (int)vt_ld; ex.col2 = 2 * Cp;
        TRY(add_linear(prog_frame, tokens(hs), f.w, 3 * Cp, C, f.bias, qk.p, 2 * Cp, nullptr, 0, 0, -1, &ex));
    } else {
        Act ln = new_act(B, x.h, x.w, C);
        TRY(add_layernorm(hs, t + "norm1", ln));
        __half* wqk = pack_rows(t + "attn1.qk", {{t + "attn1.to_q.weight", head_perm(0)}, {t + "attn1.to_k.weight", head_perm(0)}}, C, s);
        __half* wv = pack_rows(t + "attn1.v", {{t + "attn1.to_v.weight", head_perm(0)}}, C, s);
        if (!wqk || !wv) return -1;
        TRY(add_linear(prog_frame, tokens(ln), wqk, 2 * Cp, C, nullptr, qk.p, 2 * Cp, nullptr, 0));
        // V^T = Wv . ln^T : weights on the M side, tokens on the N side.  TMA needs the per-batch column origin
        // 16-byte aligned, so when HW is not a multiple of 8 each batch item gets its own padded column range.
        allow_swap = false;  // V^T already has the weights on the M side
        for (int bi = 0; bi < (one_gemm ? 1 : B); ++bi) {
            ActView wv_view{wv, 1, 1, Cp, C, C};
            IgemmDesc d{};
            d.nseg = 1; d.src[0] = wv_view; d.ntap[0] = 1;
            d.w = one_gemm ? ln.p : ln.p + (long)bi * HW * ln.ld;
            d.w_rows = one_gemm ? (int)M : HW; d.w_ld = C; d.stride = 1;
            d.Nb = 1; d.Ho = 1; d.Wo = Cp;
            d.epi.out = one_gemm ? vt : vt + (long)bi * HWp;
            d.epi.ldc = (int)vt_ld; d.epi.acc_scale = 1.f; d.epi.res_scale = 1.f;
            d.epi.n_valid = one_gemm ? (int)M : HW;
            TRY(add_igemm(prog_frame, d));
        }
        allow_swap = true;
    }
    Act ao = new_act(B, x.h, x.w, C);
    {
        AttnDesc a{};
        a.q = qk.p; a.ldq = 2 * Cp;
        a.k = qk.p + Cp; a.ldk = 2 * Cp; a.k_bstride = HW; a.k_rows = M;
        a.vt = vt; a.ldvt = (int)vt_ld; a.vt_bstride = vt_bstride; a.vt_cols = one_gemm ? M : (long)B * HWp;
        a.out = ao.p; a.ldo = C;
        a.nb = B; a.heads = heads; a.sq = HW; a.skv = HW; a.d_real = d_real; a.dp = dp;
        AttnPlan plan;
        TRY(attn_plan(a, &plan));
        ++launches;
        prog_frame.push_back(Op([plan](cudaStream_t st) { return attn_launch(plan, st); }, "attn " + p,
                               4.0 * a.nb * a.heads * (double)a.sq * a.skv * a.d_real));
    }
    const Raw* wo1 = get(t + "attn1.to_out.0.weight");
    if (!wo1) return -1;
    Act hs2 = new_act(B, x.h, x.w, C);
    {
        LinExtra ex; ex.rowstat_out = st2;
        TRY(add_linear(prog_frame, tokens(ao), wo1->p, C, C, vec({t + "attn1.to_out.0.bias"}), hs2.p, C, hs.p, C, 0, -1, &ex));
    }
    // ---- cross attention against the cached prompt K / V^T
    __half* wk2 = pack_rows(t + "attn2.k", {{t + "attn2.to_k.weight", head_perm(0)}}, D, s);
    __half* wv2 = pack_rows(t + "attn2.v", {{t + "attn2.to_v.weight", head_perm(0)}}, D, s);
    if (!wk2 || !wv2) return -1;
    const int Lpad = 128 * ((L + 127) / 128);
    // One prompt for every batch item, or (a guided batch with unconditional rows) one Lpad-row context per batch item: uncond
    // or cond embeddings, zero padded, addressed by the attention's per-batch K / V^T strides.  Either way the K / V^T
    // GEMMs run once per prompt (prog_prompt), not per frame.
    const bool per_row = uc_rows > 0;
    const int ctx_n = per_row ? B * Lpad : L;   // context rows of the K / V^T GEMMs
    const int vt_ld2 = per_row ? B * Lpad : Lpad;
    __half* kc = static_cast<__half*>(prog.alloc((size_t)ctx_n * Cp * 2));
    __half* vct = static_cast<__half*>(prog.alloc((size_t)Cp * vt_ld2 * 2));
    if (!kc || !vct) return -1;
    {
        allow_swap = false;
        const __half* cp = per_row ? ctx_rows : ctx;
        ActView ctxv{cp, 1, 1, ctx_n, D, D};
        TRY(add_linear(prog_prompt, ctxv, wk2, Cp, D, nullptr, kc, Cp, nullptr, 0));
        ActView wvv{wv2, 1, 1, Cp, D, D};
        IgemmDesc d{};
        d.nseg = 1; d.src[0] = wvv; d.ntap[0] = 1;
        d.w = cp; d.w_rows = ctx_n; d.w_ld = D; d.stride = 1;
        d.Nb = 1; d.Ho = 1; d.Wo = Cp;
        d.epi.out = vct; d.epi.ldc = vt_ld2; d.epi.acc_scale = 1.f; d.epi.res_scale = 1.f; d.epi.n_valid = ctx_n;
        TRY(add_igemm(prog_prompt, d));
        allow_swap = true;
    }
    Act q2 = new_act(1, 1, (int)M, Cp);
    if (fold) {
        LnFold f;
        TRY(fold_ln(t + "attn2.q+ln", {{t + "attn2.to_q.weight", head_perm(0)}}, C, t + "norm2", nullptr, &f, s));
        LinExtra ex; ex.rowstat_in = st2; ex.colsum = f.colsum; ex.ln_c = C;
        TRY(add_linear(prog_frame, tokens(hs2), f.w, Cp, C, f.bias, q2.p, Cp, nullptr, 0, 0, -1, &ex));
    } else {
        Act ln2 = new_act(B, x.h, x.w, C);
        TRY(add_layernorm(hs2, t + "norm2", ln2));
        __half* wq2 = pack_rows(t + "attn2.q", {{t + "attn2.to_q.weight", head_perm(0)}}, C, s);
        if (!wq2) return -1;
        TRY(add_linear(prog_frame, tokens(ln2), wq2, Cp, C, nullptr, q2.p, Cp, nullptr, 0));
    }
    Act ao2 = new_act(B, x.h, x.w, C);
    {
        AttnDesc a{};
        a.q = q2.p; a.ldq = Cp;
        a.k = kc; a.ldk = Cp; a.k_bstride = per_row ? Lpad : 0; a.k_rows = ctx_n;
        a.vt = vct; a.ldvt = vt_ld2; a.vt_bstride = per_row ? Lpad : 0; a.vt_cols = ctx_n;
        a.out = ao2.p; a.ldo = C;
        a.nb = B; a.heads = heads; a.sq = HW; a.skv = L; a.d_real = d_real; a.dp = dp;
        AttnPlan plan;
        TRY(attn_plan(a, &plan));
        ++launches;
        prog_frame.push_back(Op([plan](cudaStream_t st) { return attn_launch(plan, st); }, "attn " + p,
                               4.0 * a.nb * a.heads * (double)a.sq * a.skv * a.d_real));
    }
    const Raw* wo2 = get(t + "attn2.to_out.0.weight");
    if (!wo2) return -1;
    Act hs3 = new_act(B, x.h, x.w, C);
    {
        LinExtra ex; ex.rowstat_out = st3;
        TRY(add_linear(prog_frame, tokens(ao2), wo2->p, C, C, vec({t + "attn2.to_out.0.bias"}), hs3.p, C, hs2.p, C, 0, -1, &ex));
    }
    // ---- GEGLU feed-forward
    Act ff = new_act(1, 1, (int)M, inner);
    {
        IgemmDesc d{};
        d.nseg = 1; d.ntap[0] = 1;
        d.w_rows = 2 * inner; d.w_ld = C; d.stride = 1;
        d.Nb = 1; d.Ho = 1; d.Wo = (int)M;
        d.BN = 128;   // the 128-column value/gate interleave of the packed rows
        d.epi.out = ff.p; d.epi.ldc = inner; d.epi.acc_scale = 1.f; d.epi.res_scale = 1.f;
        d.epi.flags = IG_GEGLU; d.epi.n_valid = inner;
        if (fold) {
            LnFold f;
            TRY(fold_ln(t + "ff1+ln", {{t + "ff.net.0.proj.weight", gperm}}, C, t + "norm3", bff1, &f, s));
            d.src[0] = tokens(hs3);
            d.w = f.w; d.epi.colbias = f.bias;
            d.epi.rowstat_in = st3; d.epi.colsum = f.colsum; d.epi.ln_inv_c = 1.f / (float)C; d.epi.ln_eps = 1e-5f;
        } else {
            Act ln3 = new_act(B, x.h, x.w, C);
            TRY(add_layernorm(hs3, t + "norm3", ln3));
            __half* wff1 = pack_rows(t + "ff1", {{t + "ff.net.0.proj.weight", gperm}}, C, s);
            if (!wff1) return -1;
            d.src[0] = tokens(ln3);
            d.w = wff1; d.epi.colbias = bff1;
        }
        IgemmPlan plan;
        TRY(igemm_plan(d, &plan));
        push_igemm(prog_frame, plan, "igemm geglu " + p, 2.0 * (double)M * (2.0 * inner) * C);
    }
    const Raw* wff2 = get(t + "ff.net.2.weight");
    if (!wff2) return -1;
    Act hs4 = new_act(B, x.h, x.w, C);
    TRY(add_linear(prog_frame, tokens(ff), wff2->p, C, inner, vec({t + "ff.net.2.bias"}), hs4.p, C, hs3.p, C));
    // proj_out + residual with the block input
    const Raw* wpo = get(p + "proj_out.weight");
    if (!wpo) return -1;
    *out = new_act(B, x.h, x.w, C);
    return add_linear(prog_frame, tokens(hs4), wpo->p, C, C, vec({p + "proj_out.bias"}), out->p, C, x.p, x.ld);
}

// AutoencoderTinyBlock: relu(conv(relu(conv(relu(conv(x))))) + x)
int b2sd_engine::build_taesd_block(const std::string& p, const Act& x, Act* out, cudaStream_t s) {
    cur = p;
    allow_swap = false;
    Act a = new_act(x.n, x.h, x.w, x.c), b = new_act(x.n, x.h, x.w, x.c);
    *out = new_act(x.n, x.h, x.w, x.c);
    TRY(add_conv(prog_frame, x, p + ".conv.0.weight", p + ".conv.0.bias", 9, 1, a, IG_RELU, nullptr, s));
    TRY(add_conv(prog_frame, a, p + ".conv.2.weight", p + ".conv.2.bias", 9, 1, b, IG_RELU, nullptr, s));
    return add_conv(prog_frame, b, p + ".conv.4.weight", p + ".conv.4.bias", 9, 1, *out, IG_RELU, &x, s);
}

int b2sd_engine::build_program(cudaStream_t s) {
    prog.reset();
    prog_frame.clear(); prog_prompt.clear(); prog_time.clear();
    taps.clear();
    launches = 0;
    drop_graphs();
    const int T = cfg.batch, B = unet_rows(), H = cfg.height, W = cfg.width;   // B: UNet batch (T + unconditional rows)
    const int* ch = cfg.block_out_channels;
    const int nlev = 4;
    {
        // LayerNorm row statistics of every transformer block (3 per block, [tokens][2] 64-bit words), one slab that a single
        // memset node clears at the start of each frame
        long words = 0;
        for (int i = 0; i < nlev; ++i) {
            const long tokens_i = (long)B * (lh >> i) * (lw >> i);
            const int blocks_i = (cfg.down_attn[i] ? cfg.layers_per_block + (cfg.layers_per_block + 1) : 0) + (i == nlev - 1 ? 1 : 0);
            words += 3 * 2 * tokens_i * blocks_i;
        }
        ln_stats_cap = (size_t)words;
        ln_stats_used = 0;
        ln_stats = static_cast<unsigned long long*>(prog.alloc(ln_stats_cap * sizeof(unsigned long long)));
        if (!ln_stats) return -1;
    }
    ctx_rows = nullptr;
    if (uc_rows > 0) {
        // per-row prompt contexts of the guided batch, refreshed from uctx / ctx by the prompt program (b2sd_set_prompt_embeds)
        const int L = cfg.ctx_tokens, D = cfg.cross_attention_dim, Lpad = 128 * ((L + 127) / 128);
        ctx_rows = static_cast<__half*>(prog.alloc((size_t)B * Lpad * D * 2));
        if (!ctx_rows) return -1;
        CUDA_OK(cudaMemsetAsync(ctx_rows, 0, (size_t)B * Lpad * D * 2, s));   // padding rows: K = V = 0, masked by skv
        __half* dst = ctx_rows; const __half* cond = ctx; const __half* unc = uctx; const int ucr = uc_rows;
        prog_prompt.push_back(Op([=](cudaStream_t st) {
            for (int r = 0; r < B; ++r)
                if (cudaMemcpyAsync(dst + (size_t)r * Lpad * D, r < ucr ? unc : cond, (size_t)L * D * 2, cudaMemcpyDeviceToDevice, st) !=
                    cudaSuccess) { b2_set_error("copy of the per-row prompt contexts failed"); return -1; }
            return 0; }, "ctx rows"));
    }

    allow_swap = false;
    // ================= TAESD encoder (EncoderTiny) =================
    Act e = new_act(1, H, W, 64);
    {
        head = SmallConvArgs{};
        head.wt = small_w("vae.encoder.layers.0.weight", s);
        if (!head.wt) return -1;
        head.bias = vec({"vae.encoder.layers.0.bias"});
        head.y = e.p; head.ldy = e.ld; head.nb = 1; head.h = H; head.w_ = W; head.cin = 3; head.cout = 64;
        head.flags = SC_IN_U8;
        if (!head.bias) return -1;
        ++launches;
    }
    int li = 1;
    const int enc_blocks[4] = {1, 3, 3, 3};
    for (int st = 0; st < 4; ++st) {
        if (st > 0) {
            Act dwn = new_act(1, e.h / 2, e.w / 2, 64);
            TRY(add_conv(prog_frame, e, "vae.encoder.layers." + std::to_string(li) + ".weight", "", 9, 2, dwn, 0, nullptr, s));
            e = dwn;
            ++li;
        }
        for (int k = 0; k < enc_blocks[st]; ++k) {
            Act o;
            TRY(build_taesd_block("vae.encoder.layers." + std::to_string(li), e, &o, s));
            e = o;
            ++li;
        }
    }
    {
        // latent head + StreamDiffusion.encode_image add-noise: x_t = alpha0 * z + beta0 * init_noise[0]
        Act xt;  // slot 0 of the UNet input batch
        xt.p = x_in.p; xt.n = 1; xt.h = lh; xt.w = lw; xt.c = 4; xt.ld = 4;
        Act nz = xt;
        nz.p = noise;
        const std::string k = "vae.encoder.layers." + std::to_string(li);
        idx_enc_end = prog_frame.size();   // everything before this conv only touches this engine's own activations
        TRY(add_conv(prog_frame, e, k + ".weight", k + ".bias", 9, 1, xt, 0, &nz, s, coef_host[0][0], coef_host[1][0]));
        taps["x_t"] = xt;
    }
    taps["unet_in"] = x_in;

    allow_swap = true;
    // ================= UNet2DConditionModel =================
    Act h = new_act(B, lh, lw, ch[0]);
    {
        SmallConvArgs a{};
        a.wt = small_w("conv_in.weight", s);
        if (!a.wt) return -1;
        a.x = x_in.p; a.bias = vec({"conv_in.bias"});
        a.y = h.p; a.ldy = h.ld; a.nb = B; a.h = lh; a.w_ = lw; a.cin = 4; a.cout = ch[0]; a.in_h = lh; a.in_w = lw;
        a.uc_rows = uc_rows;   // UNet input = cat(x[0:uc_rows], x): gathered here, never copied
        if (!a.bias) return -1;
        ++launches;
        prog_frame.push_back(Op([a](cudaStream_t st) { return smallconv_launch(a, st); }, "smallconv"));
    }
    taps["conv_in"] = h;
    std::vector<Act> skips{h};
    for (int i = 0; i < nlev; ++i) {
        for (int j = 0; j < cfg.layers_per_block; ++j) {
            Act o;
            const std::string bp = "down_blocks." + std::to_string(i);
            TRY(build_resnet(bp + ".resnets." + std::to_string(j) + ".", h, nullptr, ch[i], &o, s));
            h = o;
            if (cfg.down_attn[i]) {
                TRY(build_transformer(bp + ".attentions." + std::to_string(j) + ".", h, cfg.heads[i], &o, s));
                h = o;
            }
            skips.push_back(h);
            taps["down." + std::to_string(i) + "." + std::to_string(j)] = h;
        }
        if (i != nlev - 1) {
            Act o = new_act(B, h.h / 2, h.w / 2, ch[i]);
            const std::string k = "down_blocks." + std::to_string(i) + ".downsamplers.0.conv.";
            TRY(add_conv(prog_frame, h, k + "weight", k + "bias", 9, 2, o, 0, nullptr, s));
            h = o;
            skips.push_back(h);
        }
    }
    {
        Act o;
        TRY(build_resnet("mid_block.resnets.0.", h, nullptr, ch[nlev - 1], &o, s)); h = o;
        TRY(build_transformer("mid_block.attentions.0.", h, cfg.heads[nlev - 1], &o, s)); h = o;
        TRY(build_resnet("mid_block.resnets.1.", h, nullptr, ch[nlev - 1], &o, s)); h = o;
        taps["mid"] = h;
    }
    for (int i = 0; i < nlev; ++i) {
        const int co = ch[nlev - 1 - i];
        const int hd = cfg.heads[nlev - 1 - i];
        const bool attn = cfg.down_attn[nlev - 1 - i] != 0;
        for (int j = 0; j < cfg.layers_per_block + 1; ++j) {
            Act sk = skips.back();
            skips.pop_back();
            Act o;
            const std::string bp = "up_blocks." + std::to_string(i);
            TRY(build_resnet(bp + ".resnets." + std::to_string(j) + ".", h, &sk, co, &o, s));
            h = o;
            if (attn) {
                TRY(build_transformer(bp + ".attentions." + std::to_string(j) + ".", h, hd, &o, s));
                h = o;
            }
            taps["up." + std::to_string(i) + "." + std::to_string(j)] = h;
        }
        if (i != nlev - 1) {
            Act up = new_act(B, h.h * 2, h.w * 2, co);
            const Act hin = h;
            ++launches;
            prog_frame.push_back(Op([hin, up](cudaStream_t st) { return upsample2x_launch(hin.p, up.p, hin.n, hin.h, hin.w, hin.c, st); }, "upsample2x"));
            Act o = new_act(B, up.h, up.w, co);
            const std::string k = "up_blocks." + std::to_string(i) + ".upsamplers.0.conv.";
            TRY(add_conv(prog_frame, up, k + "weight", k + "bias", 9, 1, o, 0, nullptr, s));
            h = o;
        }
    }
    Act nout = new_act(B, lh, lw, ch[0]);
    TRY(add_groupnorm(h, nullptr, "conv_norm_out", nout, 1e-5f, 1));
    Act eps = new_act(B, lh, lw, 4);
    TRY(add_conv(prog_frame, nout, "conv_out.weight", "conv_out.bias", 9, 1, eps, 0, nullptr, s));
    taps["eps"] = eps;
    // ================= scheduler_step_batch + stream-batch buffer update =================
    Act x0 = new_act(1, lh, lw, 4);
    {
        __half* xp = x_in.p; const __half* ep = eps.p; const __half* np_ = noise; const float* cf = coef; __half* op = x0.p;
        const int hw = lh * lw, dan = cfg.do_add_noise;
        ++launches;
        if (guide.cfg_type == B2SD_CFG_NONE) {
            prog_frame.push_back(Op([=](cudaStream_t st) { return lcm_step_launch(xp, ep, np_, cf, op, T, hw, dan, st); }, "lcm_step"));
        } else {
            __half* sp = stock; const int ct = guide.cfg_type; const float g = guide.scale, dl = guide.delta;
            prog_frame.push_back(Op([=](cudaStream_t st) { return lcm_cfg_step_launch(xp, ep, np_, sp, cf, op, T, hw, dan, ct, g, dl, st); },
                                    "lcm_cfg_step"));
        }
        idx_unet_end = prog_frame.size();
    }
    taps["x0"] = x0;
    {
        Act sn;
        sn.p = stock; sn.n = T; sn.h = lh; sn.w = lw; sn.c = 4; sn.ld = 4;
        taps["stock_noise"] = sn;
    }
    allow_swap = false;
    // ================= TAESD decoder (DecoderTiny) =================
    Act dcur = new_act(1, lh, lw, 64);
    {
        SmallConvArgs a{};
        a.wt = small_w("vae.decoder.layers.0.weight", s);
        if (!a.wt) return -1;
        a.x = x0.p; a.bias = vec({"vae.decoder.layers.0.bias"});
        a.y = dcur.p; a.ldy = dcur.ld; a.nb = 1; a.h = lh; a.w_ = lw; a.cin = 4; a.cout = 64; a.in_h = lh; a.in_w = lw;
        a.flags = SC_IN_TANH3 | SC_OUT_RELU;
        if (!a.bias) return -1;
        ++launches;
        prog_frame.push_back(Op([a](cudaStream_t st) { return smallconv_launch(a, st); }, "smallconv"));
    }
    li = 2;
    const int dec_blocks[4] = {3, 3, 3, 1};
    for (int st = 0; st < 4; ++st) {
        for (int k = 0; k < dec_blocks[st]; ++k) {
            Act o;
            TRY(build_taesd_block("vae.decoder.layers." + std::to_string(li), dcur, &o, s));
            dcur = o;
            ++li;
        }
        if (st != 3) {
            Act up = new_act(1, dcur.h * 2, dcur.w * 2, 64);
            const Act hin = dcur;
            ++launches;
            prog_frame.push_back(Op([hin, up](cudaStream_t s2) { return upsample2x_launch(hin.p, up.p, hin.n, hin.h, hin.w, hin.c, s2); }, "upsample2x"));
            ++li;  // nn.Upsample
            Act o = new_act(1, up.h, up.w, 64);
            TRY(add_conv(prog_frame, up, "vae.decoder.layers." + std::to_string(li) + ".weight", "", 9, 1, o, 0, nullptr, s));
            dcur = o;
            ++li;
        } else {
            image = new_act(1, H, W, 3, 8);
            const std::string k = "vae.decoder.layers." + std::to_string(li);
            TRY(add_conv(prog_frame, dcur, k + ".weight", k + ".bias", 9, 1, image, 0, nullptr, s));
        }
    }
    taps["image"] = image;
    ++launches;  // post_u8 tail
    if (ln_stats_used) {
        unsigned long long* sp = ln_stats;
        const size_t bytes = ln_stats_used * sizeof(unsigned long long);
        // first op of the UNet stage (the statistics belong to the transformer blocks)
        prog_frame.insert(prog_frame.begin() + idx_enc_end, Op([sp, bytes](cudaStream_t st) {
            if (cudaMemsetAsync(sp, 0, bytes, st) != cudaSuccess) { b2_set_error("memset of the LayerNorm statistics failed"); return -1; }
            return 0; }, "memset ln_stats"));
        idx_unet_end += 1;
    }
    CUDA_OK(cudaStreamSynchronize(s));
    built = true;
    return 0;
}

// ================================================================================================
extern "C" {

static int create_engine(const b2sd_config* cfg, std::shared_ptr<WeightStore> store, b2sd_handle* out);
static int alloc_unet_rows(b2sd_handle e, int rows);

int b2sd_create(const b2sd_config* cfg, b2sd_handle* out) { return create_engine(cfg, std::make_shared<WeightStore>(), out); }

/* A second engine over the SAME parameters (shared weight store): its own activations, stream state and CUDA graph, so two
 * frames can be in flight on two CUDA streams.  cfg may differ from the parent's in batch / size only. */
int b2sd_create_lane(b2sd_handle parent, const b2sd_config* cfg, b2sd_handle* out) {
    if (!parent) {
        b2_set_error("b2sd_create_lane: null parent");
        return -1;
    }
    b2sd_config c = cfg ? *cfg : parent->cfg;
    for (int i = 0; i < 4; ++i)
        if (c.block_out_channels[i] != parent->cfg.block_out_channels[i] || c.heads[i] != parent->cfg.heads[i] ||
            c.down_attn[i] != parent->cfg.down_attn[i]) {
            b2_set_error("b2sd_create_lane: the lane's architecture differs from its parent's");
            return -1;
        }
    if (create_engine(&c, parent->ws, out)) return -1;
    (*out)->concurrency = parent->concurrency > 1 ? parent->concurrency : 2;
    return 0;
}

static int create_engine(const b2sd_config* cfg, std::shared_ptr<WeightStore> store, b2sd_handle* out) {
    if (!cfg || !out) {
        b2_set_error("b2sd_create: null argument");
        return -1;
    }
    if (cfg->height % 64 || cfg->width % 64 || cfg->batch < 1 || cfg->batch > 16) {
        b2_set_error("b2sd_create: height/width must be multiples of 64, 1 <= batch <= 16 (got %dx%d, %d)",
                     cfg->height, cfg->width, cfg->batch);
        return -1;
    }
    for (int i = 0; i < 4; ++i) {
        if (cfg->block_out_channels[i] % 64 || cfg->heads[i] < 1 || cfg->block_out_channels[i] % cfg->heads[i]) {
            b2_set_error("b2sd_create: block_out_channels must be multiples of 64 and divisible by heads");
            return -1;
        }
    }
    if (cfg->cross_attention_dim % 64) {
        b2_set_error("b2sd_create: cross_attention_dim must be a multiple of 64");
        return -1;
    }
    int dev = 0;
    cudaDeviceProp prop;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaGetDeviceProperties(&prop, dev) != cudaSuccess) {
        b2_set_error("b2sd_create: no CUDA device (this library has no CPU path)");
        return -1;
    }
    if (prop.major != 10) {
        b2_set_error("b2sd_create: device sm_%d%d is not Blackwell sm_100 (kernels are sm_100a only)", prop.major, prop.minor);
        return -1;
    }
    if (igemm_init() || attn_init() || tconv_init()) return -1;
    b2sd_engine* e = new b2sd_engine(std::move(store));
    e->cfg = *cfg;
    e->lh = cfg->height / 8;
    e->lw = cfg->width / 8;
    const int B = cfg->batch;
    e->x_in.n = B; e->x_in.h = e->lh; e->x_in.w = e->lw; e->x_in.c = 4; e->x_in.ld = 4;
    e->x_in.p = static_cast<__half*>(e->state.alloc((size_t)e->x_in.elems() * 2));
    e->noise = static_cast<__half*>(e->state.alloc((size_t)e->x_in.elems() * 2));
    e->stock = static_cast<__half*>(e->state.alloc((size_t)e->x_in.elems() * 2));
    e->coef = static_cast<float*>(e->state.alloc(4 * B * sizeof(float)));
    e->ctx = static_cast<__half*>(e->state.alloc((size_t)cfg->ctx_tokens * cfg->cross_attention_dim * 2));
    e->uctx = static_cast<__half*>(e->state.alloc((size_t)cfg->ctx_tokens * cfg->cross_attention_dim * 2));
    e->tile_counters = static_cast<int*>(e->state.alloc(65536 * sizeof(int)));
    if (e->tile_counters) cudaMemset(e->tile_counters, 0, 65536 * sizeof(int));
    if (e->stock) cudaMemset(e->stock, 0, (size_t)e->x_in.elems() * 2);
    if (!e->x_in.p || !e->noise || !e->stock || !e->coef || !e->ctx || !e->uctx || alloc_unet_rows(e, B)) {
        b2_set_error("b2sd_create: cudaMalloc failed");
        delete e;
        return -1;
    }
    *out = e;
    return 0;
}

int b2sd_destroy(b2sd_handle h) {
    if (h) {
        cudaDeviceSynchronize();
        delete h;
    }
    return 0;
}

// Parameters whose raw layout no kernel reads: they are re-laid-out once by pack_conv / pack_rows / small_w.
static bool is_pack_only(const std::string& key, const int64_t* shape, int ndim) {
    auto has = [&](const char* t) { return key.find(t) != std::string::npos; };
    if (ndim == 4 && shape[2] == 3) return true;                       // every 3x3 convolution (incl. the Cin <= 4 ones)
    if (ndim == 4 && has("conv_shortcut.weight")) return true;         // packed into the conv2 rows
    if (ndim == 2 && (has(".to_q.weight") || has(".to_k.weight") || has(".to_v.weight"))) return true;   // per-head gather
    if (ndim == 2 && has("ff.net.0.proj.weight")) return true;         // GEGLU value/gate interleave
    return false;
}

int b2sd_load_tensor(b2sd_handle h, const char* key, const void* ptr, int dtype, const int64_t* shape, int ndim) {
    if (!h || !key || !ptr || ndim < 1 || ndim > 4) {
        b2_set_error("b2sd_load_tensor: bad argument");
        return -1;
    }
    Raw r;
    r.shape.assign(shape, shape + ndim);
    const long n = r.numel();
    if (h->raw_released) {
        b2_set_error("b2sd_load_tensor(%s): the pack-only raw weights were released after b2sd_prepare; create a new engine to "
                     "load different parameters (or set B2_KEEP_RAW=1 before the first prepare)", key);
        return -1;
    }
    r.pack_only = is_pack_only(key, shape, ndim);
    auto old = h->raw.find(key);
    if (old != h->raw.end()) {
        // Reload of a parameter (e.g. a LoRA swap): everything derived from the old values is stale.  The packed / fp32
        // caches are keyed by parameter name, so drop them all (they are rebuilt by the next b2sd_prepare); a same-shape
        // reload overwrites the device copy in place instead of growing the bump arena.
        h->packed.clear(); h->packed_bytes.clear();
        h->fvec.clear(); h->fvec_bytes.clear();
        if (old->second.shape == r.shape) r.p = old->second.p;
    }
    if (!r.p) r.p = static_cast<__half*>((r.pack_only ? h->raw_only : h->weights).alloc((size_t)n * 2));
    if (!r.p) {
        b2_set_error("b2sd_load_tensor: cudaMalloc failed for %s", key);
        return -1;
    }
    if (dtype == 0) {
        CUDA_OK(cudaMemcpy(r.p, ptr, (size_t)n * 2, cudaMemcpyDefault));
    } else if (dtype == 1) {
        float* tmp = nullptr;
        CUDA_OK(cudaMalloc(&tmp, (size_t)n * 4));
        cudaError_t e1 = cudaMemcpy(tmp, ptr, (size_t)n * 4, cudaMemcpyDefault);
        int rc = (e1 == cudaSuccess) ? cast_f32_to_f16_launch(tmp, r.p, n, 0) : -1;
        cudaDeviceSynchronize();
        cudaFree(tmp);
        if (rc) {
            b2_set_error("b2sd_load_tensor: upload of %s failed", key);
            return -1;
        }
    } else {
        b2_set_error("b2sd_load_tensor: dtype %d", dtype);
        return -1;
    }
    if (ndim == 1) {
        std::vector<__half> hh(n);
        CUDA_OK(cudaMemcpy(hh.data(), r.p, (size_t)n * 2, cudaMemcpyDeviceToHost));
        r.host.resize(n);
        for (long i = 0; i < n; ++i) r.host[i] = __half2float(hh[i]);
    }
    h->raw[key] = std::move(r);
    h->built = false;
    return 0;
}

// Per-UNet-row state (timesteps, time embeddings, GroupNorm workspace) for `rows` rows; grows only (bump arena).
static int alloc_unet_rows(b2sd_handle e, int rows) {
    if (rows <= e->rows_cap) return 0;
    const int C0 = e->cfg.block_out_channels[0];
    e->tsteps = static_cast<float*>(e->state.alloc(rows * sizeof(float)));
    e->temb_sin = static_cast<float*>(e->state.alloc((size_t)rows * C0 * sizeof(float)));
    e->temb_h = static_cast<float*>(e->state.alloc((size_t)rows * 4 * C0 * sizeof(float)));
    e->temb = static_cast<float*>(e->state.alloc((size_t)rows * 4 * C0 * sizeof(float)));
    e->gn_ws = static_cast<float*>(e->state.alloc(groupnorm_partial_floats(rows, e->cfg.norm_groups) * sizeof(float)));
    if (!e->tsteps || !e->temb_sin || !e->temb_h || !e->temb || !e->gn_ws) {
        b2_set_error("cudaMalloc of the per-row UNet state (%d rows) failed", rows);
        return -1;
    }
    e->rows_cap = rows;
    return 0;
}

// sub_timesteps [T] -> tsteps of the UNet rows: row r < uc_rows takes t[r], row r >= uc_rows takes t[r - uc_rows]
static int upload_timesteps(b2sd_handle h, const float* timesteps, cudaStream_t s) {
    const int rows = h->unet_rows(), u = h->uc_rows;
    std::vector<float> t(rows);
    for (int r = 0; r < rows; ++r) t[r] = timesteps[r < u ? r : r - u];
    CUDA_OK(cudaMemcpyAsync(h->tsteps, t.data(), rows * sizeof(float), cudaMemcpyHostToDevice, s));
    CUDA_OK(cudaStreamSynchronize(s));
    return 0;
}

static int refresh_time(b2sd_handle h, cudaStream_t s) {
    const int B = h->unet_rows(), C0 = h->cfg.block_out_channels[0], TD = 4 * C0;
    const Raw* w1 = h->get("time_embedding.linear_1.weight");
    const Raw* w2 = h->get("time_embedding.linear_2.weight");
    const float* b1 = h->vec({"time_embedding.linear_1.bias"});
    const float* b2v = h->vec({"time_embedding.linear_2.bias"});
    if (!w1 || !w2 || !b1 || !b2v) return -1;
    TRY(timestep_embedding_launch(h->tsteps, h->temb_sin, B, C0, s));
    TRY(small_linear_launch(h->temb_sin, C0, w1->p, b1, h->temb_h, TD, B, TD, C0, 0, s));
    TRY(small_linear_launch(h->temb_h, TD, w2->p, b2v, h->temb, TD, B, TD, TD, 1, s));
    return h->run(h->prog_time, s);
}

int b2sd_prepare(b2sd_handle h, const void* prompt_embeds, const float* timesteps, const float* coef,
                 const void* init_noise, void* stream) {
    if (!h || !prompt_embeds || !timesteps || !coef || !init_noise) {
        b2_set_error("b2sd_prepare: null argument");
        return -1;
    }
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    const int B = h->cfg.batch, lh = h->lh, lw = h->lw;
    // guidance requested by b2sd_set_guidance takes effect here
    const b2sd_engine::Guidance& g = h->guide_req;
    const bool guided = g.cfg_type != B2SD_CFG_NONE && g.scale > 1.f;
    const int uc = !guided ? 0 : (g.cfg_type == B2SD_CFG_INITIALIZE ? 1 : (g.cfg_type == B2SD_CFG_FULL ? B : 0));
    if (B + uc > 16) {
        b2_set_error("b2sd_prepare: the guided UNet batch of %d rows exceeds 16", B + uc);
        return -1;
    }
    if (uc > 0 && h->uncond_host.empty()) {
        b2_set_error("b2sd_prepare: cfg_type initialize / full needs the unconditional embeddings (b2sd_set_guidance)");
        return -1;
    }
    TRY(alloc_unet_rows(h, B + uc));
    h->guide = guided ? g : b2sd_engine::Guidance{};
    h->uc_rows = uc;
    for (int k = 0; k < 4; ++k)
        for (int i = 0; i < B; ++i) h->coef_host[k][i] = coef[k * B + i];
    CUDA_OK(cudaMemcpyAsync(h->coef, coef, 4 * B * sizeof(float), cudaMemcpyHostToDevice, s));
    TRY(upload_timesteps(h, timesteps, s));
    CUDA_OK(cudaMemcpyAsync(h->ctx, prompt_embeds, (size_t)h->cfg.ctx_tokens * h->cfg.cross_attention_dim * 2,
                            cudaMemcpyHostToDevice, s));
    if (uc > 0)
        CUDA_OK(cudaMemcpyAsync(h->uctx, h->uncond_host.data(), h->uncond_host.size() * 2, cudaMemcpyHostToDevice, s));
    // init_noise NCHW -> NHWC (host side; once per prepare)
    {
        const __half* src = static_cast<const __half*>(init_noise);
        std::vector<__half> nhwc((size_t)B * lh * lw * 4);
        for (int b = 0; b < B; ++b)
            for (int c = 0; c < 4; ++c)
                for (int y = 0; y < lh; ++y)
                    for (int x = 0; x < lw; ++x)
                        nhwc[(((size_t)b * lh + y) * lw + x) * 4 + c] = src[(((size_t)b * 4 + c) * lh + y) * lw + x];
        CUDA_OK(cudaMemcpyAsync(h->noise, nhwc.data(), nhwc.size() * 2, cudaMemcpyHostToDevice, s));
        CUDA_OK(cudaStreamSynchronize(s));
    }
    // x_t_latent_buffer = zeros, stock_noise = zeros (StreamDiffusion.prepare); slot 0 is overwritten by every frame
    CUDA_OK(cudaMemsetAsync(h->x_in.p, 0, (size_t)h->x_in.elems() * 2, s));
    CUDA_OK(cudaMemsetAsync(h->stock, 0, (size_t)h->x_in.elems() * 2, s));
    TRY(h->build_program(s));
    TRY(h->run(h->prog_prompt, s));
    TRY(refresh_time(h, s));
    CUDA_OK(cudaStreamSynchronize(s));
    // Every pack-only parameter now exists in its kernel-native layout: drop the raw copies (about half of the UNet's
    // 1.73 GB).  Later prepares hit the packed caches and never touch them.
    static const bool keep_raw = getenv("B2_KEEP_RAW") != nullptr;
    if (!keep_raw && !h->raw_released) {
        for (auto& kv : h->raw)
            if (kv.second.pack_only) kv.second.p = nullptr;
        h->raw_only.release();
        h->raw_released = true;
    }
    return 0;
}

// ---- packed-weight blob (replaces the reference's TensorRT engine files, lib/wrapper.py:593-597, 896-910) -----------------
// Layout: "B2SDPACK" u32 version, b2sd_config, u32 count, then per entry
//   u8 kind (0 raw parameter, 1 packed fp16 matrix, 2 fp32 vector) | u32 name length | name | u32 ndim | i64 shape[ndim] |
//   u64 payload bytes (0 for a raw pack-only parameter: only its shape is needed) | payload
extern "C++" {
namespace {
struct BlobWriter {
    FILE* f;
    bool ok = true;
    void put(const void* p, size_t n) { if (ok && n && fwrite(p, 1, n, f) != n) ok = false; }
    template <class T> void pod(const T& v) { put(&v, sizeof(T)); }
    void str(const std::string& v) { pod((uint32_t)v.size()); put(v.data(), v.size()); }
};
struct BlobReader {
    FILE* f;
    bool ok = true;
    void get(void* p, size_t n) { if (ok && n && fread(p, 1, n, f) != n) ok = false; }
    template <class T> T pod() { T v{}; get(&v, sizeof(T)); return v; }
    std::string str() { uint32_t n = pod<uint32_t>(); if (!ok || n > 4096) { ok = false; return ""; } std::string v(n, 0); get(&v[0], n); return v; }
};
}  // namespace
}  // extern "C++"

int b2sd_export_packed(b2sd_handle h, const char* path) {
    if (!h || !h->built || !path) {
        b2_set_error("b2sd_export_packed: call b2sd_prepare first");
        return -1;
    }
    FILE* f = fopen(path, "wb");
    if (!f) {
        b2_set_error("b2sd_export_packed: cannot open %s", path);
        return -1;
    }
    BlobWriter w{f};
    w.put("B2SDPACK", 8);
    w.pod((uint32_t)1);
    b2sd_config cfg = h->cfg;
    cfg.batch = 0; cfg.height = 0; cfg.width = 0; cfg.use_cuda_graph = 0; cfg.do_add_noise = 0;   // the blob is independent of these
    w.pod(cfg);
    w.pod((uint32_t)(h->raw.size() + h->packed_bytes.size() + h->fvec_bytes.size()));
    std::vector<char> host;
    auto payload = [&](const void* dptr, size_t bytes) {
        w.pod((uint64_t)bytes);
        if (!bytes) return true;
        host.resize(bytes);
        if (cudaMemcpy(host.data(), dptr, bytes, cudaMemcpyDeviceToHost) != cudaSuccess) return false;
        w.put(host.data(), bytes);
        return true;
    };
    bool copy_ok = true;
    for (auto& kv : h->raw) {
        const Raw& r = kv.second;
        w.pod((uint8_t)0); w.str(kv.first);
        w.pod((uint32_t)r.shape.size());
        for (auto d : r.shape) w.pod((int64_t)d);
        copy_ok &= payload(r.p, (r.pack_only || !r.p) ? 0 : (size_t)r.numel() * 2);
    }
    for (auto& kv : h->packed_bytes) {
        w.pod((uint8_t)1); w.str(kv.first); w.pod((uint32_t)0);
        copy_ok &= payload(h->packed[kv.first], kv.second);
    }
    for (auto& kv : h->fvec_bytes) {
        w.pod((uint8_t)2); w.str(kv.first); w.pod((uint32_t)0);
        copy_ok &= payload(h->fvec[kv.first], kv.second);
    }
    const bool ok = w.ok && copy_ok && fclose(f) == 0;
    if (!ok) {
        b2_set_error("b2sd_export_packed: write to %s failed", path);
        remove(path);
        return -1;
    }
    return 0;
}

int b2sd_import_packed(b2sd_handle h, const char* path) {
    if (!h || !path) {
        b2_set_error("b2sd_import_packed: null argument");
        return -1;
    }
    if (!h->raw.empty()) {
        b2_set_error("b2sd_import_packed: the engine already holds parameters");
        return -1;
    }
    FILE* f = fopen(path, "rb");
    if (!f) {
        b2_set_error("b2sd_import_packed: cannot open %s", path);
        return -1;
    }
    BlobReader rd{f};
    char magic[8];
    rd.get(magic, 8);
    const uint32_t version = rd.pod<uint32_t>();
    b2sd_config cfg = rd.pod<b2sd_config>();
    bool same = rd.ok && memcmp(magic, "B2SDPACK", 8) == 0 && version == 1 && cfg.cross_attention_dim == h->cfg.cross_attention_dim &&
                cfg.layers_per_block == h->cfg.layers_per_block && cfg.norm_groups == h->cfg.norm_groups && cfg.ctx_tokens == h->cfg.ctx_tokens;
    for (int i = 0; i < 4 && same; ++i)
        same = cfg.block_out_channels[i] == h->cfg.block_out_channels[i] && cfg.heads[i] == h->cfg.heads[i] && cfg.down_attn[i] == h->cfg.down_attn[i];
    if (!same) {
        fclose(f);
        b2_set_error("b2sd_import_packed: %s is not a packed-weight blob of this architecture", path);
        return -1;
    }
    const uint32_t count = rd.pod<uint32_t>();
    std::vector<char> host;
    for (uint32_t i = 0; i < count && rd.ok; ++i) {
        const uint8_t kind = rd.pod<uint8_t>();
        const std::string name = rd.str();
        const uint32_t ndim = rd.pod<uint32_t>();
        Raw r;
        for (uint32_t d = 0; d < ndim && d < 8; ++d) r.shape.push_back(rd.pod<int64_t>());
        const uint64_t bytes = rd.pod<uint64_t>();
        if (!rd.ok || bytes > ((uint64_t)1 << 32)) { rd.ok = false; break; }
        void* dptr = nullptr;
        if (bytes) {
            host.resize(bytes);
            rd.get(host.data(), bytes);
            dptr = h->weights.alloc(bytes);
            if (!rd.ok || !dptr || cudaMemcpy(dptr, host.data(), bytes, cudaMemcpyHostToDevice) != cudaSuccess) { rd.ok = false; break; }
        }
        if (kind == 0) {
            r.p = static_cast<__half*>(dptr);
            r.pack_only = bytes == 0;
            if (ndim == 1 && bytes) {
                const __half* hp = reinterpret_cast<const __half*>(host.data());
                r.host.resize(bytes / 2);
                for (size_t k = 0; k < r.host.size(); ++k) r.host[k] = __half2float(hp[k]);
            }
            h->raw[name] = std::move(r);
        } else if (kind == 1) {
            h->packed[name] = static_cast<__half*>(dptr);
            h->packed_bytes[name] = bytes;
        } else if (kind == 2) {
            h->fvec[name] = static_cast<float*>(dptr);
            h->fvec_bytes[name] = bytes;
        } else {
            rd.ok = false;
        }
    }
    fclose(f);
    if (!rd.ok) {
        b2_set_error("b2sd_import_packed: %s is truncated or corrupt", path);
        return -1;
    }
    h->raw_released = true;   // there never was a raw copy of the pack-only parameters
    h->imported = true;
    h->built = false;
    return 0;
}

int b2sd_set_prompt_embeds(b2sd_handle h, const void* prompt_embeds, void* stream) {
    if (!h || !h->built) {
        b2_set_error("b2sd_set_prompt_embeds: call b2sd_prepare first");
        return -1;
    }
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    CUDA_OK(cudaMemcpyAsync(h->ctx, prompt_embeds, (size_t)h->cfg.ctx_tokens * h->cfg.cross_attention_dim * 2,
                            cudaMemcpyHostToDevice, s));
    CUDA_OK(cudaStreamSynchronize(s));
    return h->run(h->prog_prompt, s);
}

int b2sd_set_timesteps(b2sd_handle h, const float* timesteps, void* stream) {
    if (!h || !h->built) {
        b2_set_error("b2sd_set_timesteps: call b2sd_prepare first");
        return -1;
    }
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    TRY(upload_timesteps(h, timesteps, s));
    return refresh_time(h, s);
}

int b2sd_set_guidance(b2sd_handle h, int cfg_type, float guidance_scale, float delta, const void* uncond_embeds) {
    if (!h || cfg_type < B2SD_CFG_NONE || cfg_type > B2SD_CFG_FULL) {
        b2_set_error("b2sd_set_guidance: bad argument (cfg_type %d)", cfg_type);
        return -1;
    }
    if ((cfg_type == B2SD_CFG_INITIALIZE || cfg_type == B2SD_CFG_FULL) && guidance_scale > 1.f && !uncond_embeds) {
        b2_set_error("b2sd_set_guidance: cfg_type initialize / full needs the unconditional prompt embeddings");
        return -1;
    }
    h->guide_req.cfg_type = cfg_type;
    h->guide_req.scale = guidance_scale;
    h->guide_req.delta = delta;
    if (uncond_embeds) {
        const __half* src = static_cast<const __half*>(uncond_embeds);
        h->uncond_host.assign(src, src + (size_t)h->cfg.ctx_tokens * h->cfg.cross_attention_dim);
    }
    h->built = false;   // applied when the frame program is built (b2sd_prepare)
    return 0;
}

int b2sd_step(b2sd_handle h, const void* frame_in, int in_h, int in_w, void* frame_out, void* stream) {
    return b2sd_step_ex(h, frame_in, B2SD_IN_U8_NHWC, in_h, in_w, frame_out, B2SD_OUT_U8_NCHW, stream);
}

int b2sd_step_ex(b2sd_handle h, const void* frame_in, int in_kind, int in_h, int in_w, void* frame_out, int out_kind,
                 void* stream) {
    if (!h || !h->built) {
        b2_set_error("b2sd_step: call b2sd_prepare first");
        return -1;
    }
    if (!frame_in || !frame_out || in_h < 1 || in_w < 1) {
        b2_set_error("b2sd_step: bad frame arguments");
        return -1;
    }
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    SmallConvArgs a = h->head;
    a.x = frame_in; a.in_h = in_h; a.in_w = in_w;
    a.flags = in_kind == B2SD_IN_U8_NHWC ? SC_IN_U8 : (in_kind == B2SD_IN_F32_NCHW ? SC_IN_F32_NCHW : SC_IN_F16_NCHW);
    TRY(smallconv_launch(a, s));
    if (h->group) {
        // stage-pipelined lanes of one stateful stream: encoder body | [wait previous frame's UNet stage] last encoder conv,
        // UNet, scheduler step [signal] | decoder.  Lanes run on different streams; only the middle stage is serialised.
        const size_t cut[4] = {0, h->idx_enc_end, h->idx_unet_end, h->prog_frame.size()};
        for (int st = 0; st < 3; ++st) {
            if (st == 1) CUDA_OK(cudaStreamWaitEvent(s, h->group->unet_done, 0));
            if (h->cfg.use_cuda_graph) {
                if (!h->stage_exec[st]) {
                    cudaStream_t cs;
                    CUDA_OK(cudaStreamCreateWithFlags(&cs, cudaStreamNonBlocking));
                    CUDA_OK(cudaStreamBeginCapture(cs, cudaStreamCaptureModeThreadLocal));
                    int rc = h->run_range(h->prog_frame, cut[st], cut[st + 1], cs);
                    cudaError_t ec = cudaStreamEndCapture(cs, &h->stage_graph[st]);
                    cudaStreamDestroy(cs);
                    if (rc || ec != cudaSuccess || cudaGraphInstantiate(&h->stage_exec[st], h->stage_graph[st], 0) != cudaSuccess) {
                        if (!rc) b2_set_error("b2sd_step: CUDA graph capture of stage %d failed: %s", st, cudaGetErrorString(ec != cudaSuccess ? ec : cudaGetLastError()));
                        h->drop_graphs();
                        return -1;
                    }
                }
                CUDA_OK(cudaGraphLaunch(h->stage_exec[st], s));
            } else {
                TRY(h->run_range(h->prog_frame, cut[st], cut[st + 1], s));
            }
            if (st == 1) CUDA_OK(cudaEventRecord(h->group->unet_done, s));
        }
    } else if (h->cfg.use_cuda_graph) {
        if (!h->graph_exec) {
            cudaStream_t cs;
            CUDA_OK(cudaStreamCreateWithFlags(&cs, cudaStreamNonBlocking));
            CUDA_OK(cudaStreamBeginCapture(cs, cudaStreamCaptureModeThreadLocal));
            int rc = h->run(h->prog_frame, cs);
            cudaError_t ec = cudaStreamEndCapture(cs, &h->graph);
            cudaStreamDestroy(cs);
            if (rc || ec != cudaSuccess || cudaGraphInstantiate(&h->graph_exec, h->graph, 0) != cudaSuccess) {
                if (h->graph) cudaGraphDestroy(h->graph);   // a failed capture must not leave a half-built graph behind
                h->graph = nullptr;
                h->graph_exec = nullptr;
                if (!rc) b2_set_error("b2sd_step: CUDA graph capture / instantiation failed: %s", cudaGetErrorString(ec != cudaSuccess ? ec : cudaGetLastError()));
                return -1;
            }
        }
        CUDA_OK(cudaGraphLaunch(h->graph_exec, s));
    } else {
        TRY(h->run(h->prog_frame, s));
    }
    if (out_kind == B2SD_OUT_F16_NCHW)
        return post_f16_launch(h->image.p, h->image.ld, static_cast<__half*>(frame_out), 1, h->cfg.height, h->cfg.width, s);
    return post_u8_launch(h->image.p, h->image.ld, static_cast<uint8_t*>(frame_out), 1, h->cfg.height, h->cfg.width, s);
}

int b2sd_get_tensor(b2sd_handle h, const char* name, void* dst, int64_t capacity, int64_t* count, int* dims4, void* stream) {
    if (!h || !h->built || !name) {
        b2_set_error("b2sd_get_tensor: engine not prepared");
        return -1;
    }
    auto it = h->taps.find(name);
    if (it == h->taps.end()) {
        b2_set_error("b2sd_get_tensor: unknown tap '%s'", name);
        return -1;
    }
    const Act& a = it->second;
    const int64_t n = (int64_t)a.n * a.h * a.w * a.c;
    if (count) *count = n;
    if (dims4) { dims4[0] = a.n; dims4[1] = a.h; dims4[2] = a.w; dims4[3] = a.c; }
    if (!dst) return 0;
    if (capacity < n) {
        b2_set_error("b2sd_get_tensor: capacity %lld < %lld", (long long)capacity, (long long)n);
        return -1;
    }
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    CUDA_OK(cudaStreamSynchronize(s));
    CUDA_OK(cudaMemcpy2D(dst, (size_t)a.c * 2, a.p, (size_t)a.ld * 2, (size_t)a.c * 2, (size_t)a.n * a.h * a.w, cudaMemcpyDeviceToHost));
    return 0;
}

// Eager (non-graph) replay with a CUDA event after every launch: per-op device time, averaged over `iters`.
// Writes a JSON array [{"name": ..., "ms": ...}, ...] into json_buf.  Profiling aid, not the timed path.
int b2sd_profile(b2sd_handle h, const void* frame_in, int in_h, int in_w, void* frame_out, int iters, char* json_buf,
                 int64_t cap, void* stream) {
    if (!h || !h->built || !json_buf || cap < 64) {
        b2_set_error("b2sd_profile: bad arguments");
        return -1;
    }
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    const size_t nops = h->prog_frame.size() + 2;
    std::vector<cudaEvent_t> ev(nops + 1);
    for (auto& e : ev) CUDA_OK(cudaEventCreate(&e));
    std::vector<double> acc(nops, 0.0);
    SmallConvArgs a = h->head;
    a.x = frame_in; a.in_h = in_h; a.in_w = in_w; a.flags = SC_IN_U8;
    for (int it = 0; it < iters + 1; ++it) {  // first iteration is a warm-up
        CUDA_OK(cudaEventRecord(ev[0], s));
        TRY(smallconv_launch(a, s));
        CUDA_OK(cudaEventRecord(ev[1], s));
        size_t i = 1;
        for (auto& op : h->prog_frame) {
            TRY(op(s));
            ++i;
            CUDA_OK(cudaEventRecord(ev[i], s));
        }
        TRY(post_u8_launch(h->image.p, h->image.ld, static_cast<uint8_t*>(frame_out), 1, h->cfg.height, h->cfg.width, s));
        CUDA_OK(cudaEventRecord(ev[nops], s));
        CUDA_OK(cudaStreamSynchronize(s));
        if (it == 0) continue;
        for (size_t k = 0; k < nops; ++k) {
            float ms = 0.f;
            CUDA_OK(cudaEventElapsedTime(&ms, ev[k], ev[k + 1]));
            acc[k] += ms;
        }
    }
    for (auto& e : ev) cudaEventDestroy(e);
    std::string js = "[";
    char tmp[512];
    for (size_t k = 0; k < nops; ++k) {
        const char* nm = k == 0 ? "smallconv head (u8 frame -> 64ch)" : (k == nops - 1 ? "post_u8 tail" : h->prog_frame[k - 1].name.c_str());
        const double fl = (k == 0 || k == nops - 1) ? 0.0 : h->prog_frame[k - 1].flops;
        snprintf(tmp, sizeof(tmp), "%s{\"name\": \"%s\", \"ms\": %.6f, \"flops\": %.0f}", k ? ", " : "", nm, acc[k] / iters, fl);
        js += tmp;
    }
    js += "]";
    if ((int64_t)js.size() + 1 > cap) {
        b2_set_error("b2sd_profile: buffer too small (%zu needed)", js.size() + 1);
        return -1;
    }
    memcpy(json_buf, js.c_str(), js.size() + 1);
    return 0;
}

// Start gate for concurrent b2sd_profile_kind calls (one host thread per lane): every call finishes its capture / instantiation /
// warm-up replays, then waits here until all participants have arrived, so that the TIMED replays of the lanes really overlap.
static std::atomic<int> g_gate_expected{0}, g_gate_arrived{0};
int b2sd_profile_gate(int participants) {
    g_gate_arrived.store(0);
    g_gate_expected.store(participants > 1 ? participants : 0);
    return 0;
}

// Device time of one launch class inside a CUDA graph: every frame-program launch whose label starts with `kind`
// ("igemm", "attn", "groupnorm", ...) is captured, in program order, into its own graph (same PDL edges, same buffers,
// same weight streaming as the frame graph) and that graph is replayed `iters` times between two events.
int b2sd_profile_kind(b2sd_handle h, const char* kind, int iters, double* ms_per_replay, int* launches, double* flops,
                      void* stream) {
    if (!h || !h->built || !kind || iters < 1 || !ms_per_replay) {
        b2_set_error("b2sd_profile_kind: bad arguments");
        return -1;
    }
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    const std::string k(kind);
    int n = 0;
    double fl = 0.0;
    for (auto& op : h->prog_frame)   // eager pass first: one-time attribute/driver-entry-point setup may not run under capture
        if (op.name.compare(0, k.size(), k) == 0) { TRY(op(s)); ++n; fl += op.flops; }
    CUDA_OK(cudaStreamSynchronize(s));
    if (n == 0) {
        b2_set_error("b2sd_profile_kind: no launch of kind '%s'", kind);
        return -1;
    }
    cudaGraph_t g = nullptr;
    cudaGraphExec_t ge = nullptr;
    cudaStream_t cs;   // the caller's stream may be the legacy default stream, which cannot capture
    CUDA_OK(cudaStreamCreateWithFlags(&cs, cudaStreamNonBlocking));
    CUDA_OK(cudaStreamBeginCapture(cs, cudaStreamCaptureModeThreadLocal));
    int rc = 0;
    for (auto& op : h->prog_frame)
        if (op.name.compare(0, k.size(), k) == 0 && op(cs)) { rc = -1; break; }
    cudaError_t ce = cudaStreamEndCapture(cs, &g);
    cudaStreamDestroy(cs);
    if (rc || ce != cudaSuccess) {
        if (g) cudaGraphDestroy(g);
        if (!rc) b2_set_error("b2sd_profile_kind: capture failed: %s", cudaGetErrorString(ce));
        return -1;
    }
    CUDA_OK(cudaGraphInstantiate(&ge, g, 0));
    cudaEvent_t e0, e1;
    CUDA_OK(cudaEventCreate(&e0));
    CUDA_OK(cudaEventCreate(&e1));
    for (int i = 0; i < 3; ++i) CUDA_OK(cudaGraphLaunch(ge, s));
    CUDA_OK(cudaStreamSynchronize(s));
    if (const int expect = g_gate_expected.load()) {   // concurrent measurement: start the timed replays together
        g_gate_arrived.fetch_add(1);
        const auto t0 = std::chrono::steady_clock::now();
        while (g_gate_arrived.load() < expect && std::chrono::steady_clock::now() - t0 < std::chrono::seconds(20))
            std::this_thread::sleep_for(std::chrono::microseconds(50));
    }
    CUDA_OK(cudaEventRecord(e0, s));
    for (int i = 0; i < iters; ++i) CUDA_OK(cudaGraphLaunch(ge, s));
    CUDA_OK(cudaEventRecord(e1, s));
    CUDA_OK(cudaStreamSynchronize(s));
    float ms = 0.f;
    CUDA_OK(cudaEventElapsedTime(&ms, e0, e1));
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaGraphExecDestroy(ge);
    cudaGraphDestroy(g);
    *ms_per_replay = (double)ms / iters;
    if (launches) *launches = n;
    if (flops) *flops = fl;
    return 0;
}

int b2sd_launches_per_step(b2sd_handle h) { return h ? h->launches : 0; }

/* Make `lane` continue the SAME temporal stream as `owner` (both engines of one weight store, same batch and size): they
 * share the stream-batch state (x_t_latent_buffer) and are stage-pipelined -- while one lane runs the UNet stage of frame n,
 * the other runs the TAESD encoder body of frame n+1 / the decoder of frame n-1.  Frames must be submitted alternately, in
 * order, from one host thread.  Call before either engine's b2sd_prepare. */
int b2sd_share_stream_state(b2sd_handle lane, b2sd_handle owner) {
    if (!lane || !owner || lane == owner || lane->ws != owner->ws || lane->cfg.batch != owner->cfg.batch ||
        lane->cfg.height != owner->cfg.height || lane->cfg.width != owner->cfg.width) {
        b2_set_error("b2sd_share_stream_state: engines must be lanes of one weight store with the same batch and size");
        return -1;
    }
    if (!owner->group) {
        owner->group = std::make_shared<b2sd_engine::StageGroup>();
        CUDA_OK(cudaEventCreateWithFlags(&owner->group->unet_done, cudaEventDisableTiming));
    }
    lane->group = owner->group;
    lane->x_in.p = owner->x_in.p;        // the UNet input batch: slot 0 = fresh x_t, slots 1.. = x_t_latent_buffer
    lane->stock = owner->stock;          // stock_noise of residual guidance
    lane->built = false;
    owner->built = false;
    return 0;
}

int b2sd_set_concurrency(b2sd_handle h, int frames_in_flight) {
    if (!h || frames_in_flight < 1) {
        b2_set_error("b2sd_set_concurrency: bad argument");
        return -1;
    }
    h->concurrency = frames_in_flight;
    h->built = false;   // the launch policy is applied when the frame program is built (b2sd_prepare)
    return 0;
}

}  // extern "C"
