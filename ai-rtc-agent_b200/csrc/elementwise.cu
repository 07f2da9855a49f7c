// SIMT helper kernels: normalisation, resampling, tiny convolutions, scheduler step, pre/post.
#include "elementwise.cuh"

#include <stdio.h>

#include "igemm.cuh"  // b2_set_error
#include "launch.cuh"
#include "ptx.cuh"

namespace b2 {

#define B2_PDL_ENTRY()            \
    do {                          \
        pdl_launch_dependents();  \
        pdl_wait();               \
    } while (0)

#define B2_LAUNCHED(name, expr)                                            \
    do {                                                                   \
        cudaError_t e__ = (expr);                                          \
        if (e__ != cudaSuccess) {                                          \
            b2_set_error("%s launch: %s", name, cudaGetErrorString(e__));  \
            return -1;                                                     \
        }                                                                  \
    } while (0)

#define B2_CHECK_LAUNCH(name)                                              \
    do {                                                                   \
        cudaError_t e__ = cudaGetLastError();                              \
        if (e__ != cudaSuccess) {                                          \
            b2_set_error("%s launch: %s", name, cudaGetErrorString(e__));  \
            return -1;                                                     \
        }                                                                  \
    } while (0)

__device__ __forceinline__ float silu_f(float x) { return x / (1.0f + __expf(-x)); }
__device__ __forceinline__ uint64_t globaltimer_ns_ew() {
    uint64_t t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

template <typename T>
__device__ __forceinline__ T block_reduce_sum(T v, T* scratch) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    __syncthreads();
    if (lane == 0) scratch[warp] = v;
    __syncthreads();
    const int nw = (blockDim.x + 31) >> 5;
    T r = (threadIdx.x < nw) ? scratch[threadIdx.x] : T(0);
    if (warp == 0) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) r += __shfl_xor_sync(0xffffffffu, r, o);
        if (lane == 0) scratch[0] = r;
    }
    __syncthreads();
    return scratch[0];
}

// ------------------------------------------------------------------------------------------ GroupNorm
// Pass 1: grid (chunks, nb); a CTA owns `ppc` consecutive pixels x all channels (fully coalesced 16-byte
// loads), reduces per channel, then per group, and writes one (sum, sumsq) pair per (chunk, group).
// Pass 2: every CTA re-derives mean/rstd of its batch item from the <=128 chunk partials (fixed summation
// order => deterministic), then normalises 8 channels per thread.
constexpr int GN_MAX_CHUNKS = 128;

__global__ void __launch_bounds__(512) gn_stats_kernel(GroupNormArgs a, int ppc, int vc, int rpi) {
    B2_PDL_ENTRY();
    extern __shared__ float sm[];  // [rpi][C][2] then reused as [C][2]
    const int C = a.ca + a.cb;
    const int chunk = blockIdx.x, b = blockIdx.y;
    const int col = threadIdx.x % vc;       // 8-channel vector column
    const int prow = threadIdx.x / vc;      // pixel row inside one iteration
    const int c0 = col * 8;
    const bool from_a = c0 < a.ca;
    const __half* base = from_a ? a.xa + c0 : a.xb + (c0 - a.ca);
    const int ld = from_a ? a.lda : a.ldb;
    const int p_begin = chunk * ppc;
    const int p_end = min(a.hw, p_begin + ppc);
    float s[8], q[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) s[i] = q[i] = 0.f;
    if (prow < rpi) {
        for (int p = p_begin + prow; p < p_end; p += rpi) {
            const uint4 u = *reinterpret_cast<const uint4*>(base + ((long)b * a.hw + p) * ld);
            const __half2* h = reinterpret_cast<const __half2*>(&u);
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const float2 f = __half22float2(h[i]);
                s[2 * i] += f.x; q[2 * i] += f.x * f.x;
                s[2 * i + 1] += f.y; q[2 * i + 1] += f.y * f.y;
            }
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            sm[((long)prow * C + c0 + i) * 2] = s[i];
            sm[((long)prow * C + c0 + i) * 2 + 1] = q[i];
        }
    }
    __syncthreads();
    // reduce over pixel rows, then over the channels of each group
    const int cpg = C / a.groups;
    {
        // 8 lanes per group: lane `part` sums entries part, part+8, ... of the group's cpg*rpi (channel,row) pairs, then a
        // fixed 3-step shuffle tree combines the 8 parts
        const int part = threadIdx.x & 7;
        const int nent = cpg * rpi;
        for (int g = threadIdx.x >> 3; g < a.groups; g += blockDim.x >> 3) {
            float gs = 0.f, gq = 0.f;
            for (int e = part; e < nent; e += 8) {
                const int c = g * cpg + e % cpg, r = e / cpg;
                gs += sm[((long)r * C + c) * 2];
                gq += sm[((long)r * C + c) * 2 + 1];
            }
#pragma unroll
            for (int o = 4; o > 0; o >>= 1) {
                gs += __shfl_xor_sync(0xffffffffu, gs, o);
                gq += __shfl_xor_sync(0xffffffffu, gq, o);
            }
            if (part == 0)
                reinterpret_cast<float2*>(a.partial)[((long)b * a.groups + g) * GN_MAX_CHUNKS + chunk] = make_float2(gs, gq);
        }
    }
}

// mean / rstd of every group of batch item b from the per-chunk partial sums (layout [b][group][chunk]): one warp
// per group reads the chunk partials with coalesced loads (all in flight at once) and reduces them with a fixed
// shuffle tree, so the result is deterministic and costs about one L2 round trip.
__device__ __forceinline__ void gn_finalize_stats(const GroupNormArgs& a, int b, int nchunks, float* /*scratch*/,
                                                  float* s_mean, float* s_rstd) {
    const int G = a.groups;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = (blockDim.x + 31) >> 5;
    const int cpg = (a.ca + a.cb) / G;
    const float inv_n = 1.0f / ((float)a.hw * (float)cpg);
    for (int g = warp; g < G; g += nwarps) {
        const float2* src = reinterpret_cast<const float2*>(a.partial) + ((long)b * G + g) * GN_MAX_CHUNKS;
        float2 v[GN_MAX_CHUNKS / 32];
#pragma unroll
        for (int k = 0; k < GN_MAX_CHUNKS / 32; ++k)
            v[k] = (lane + 32 * k < nchunks) ? __ldcg(src + lane + 32 * k) : make_float2(0.f, 0.f);
        float gs = 0.f, gq = 0.f;
#pragma unroll
        for (int k = 0; k < GN_MAX_CHUNKS / 32; ++k) {
            gs += v[k].x;
            gq += v[k].y;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            gs += __shfl_xor_sync(0xffffffffu, gs, o);
            gq += __shfl_xor_sync(0xffffffffu, gq, o);
        }
        if (lane == 0) {
            const float mean = gs * inv_n;
            s_mean[g] = mean;
            s_rstd[g] = rsqrtf(fmaxf(gq * inv_n - mean * mean, 0.f) + a.eps);
        }
    }
    __syncthreads();
}

__global__ void __launch_bounds__(256) gn_apply_kernel(GroupNormArgs a, int nchunks, long vec_per_batch) {
    B2_PDL_ENTRY();
    __shared__ float s_mean[64], s_rstd[64];
    __shared__ float s_scratch[16 * 64 * 2];
    const int C = a.ca + a.cb;
    const int b = blockIdx.y;
    const int cpg = C / a.groups;
    gn_finalize_stats(a, b, nchunks, s_scratch, s_mean, s_rstd);
    const int vc = C / 8;
    for (long e = (long)blockIdx.x * blockDim.x + threadIdx.x; e < vec_per_batch; e += (long)gridDim.x * blockDim.x) {
        const int col = (int)(e % vc);
        const long p = e / vc;
        const int c0 = col * 8;
        const bool from_a = c0 < a.ca;
        const __half* src = from_a ? a.xa + ((long)b * a.hw + p) * a.lda + c0
                                   : a.xb + ((long)b * a.hw + p) * a.ldb + (c0 - a.ca);
        const uint4 u = *reinterpret_cast<const uint4*>(src);
        const __half2* h = reinterpret_cast<const __half2*>(&u);
        const float4 g0 = *reinterpret_cast<const float4*>(a.gamma + c0);
        const float4 g1 = *reinterpret_cast<const float4*>(a.gamma + c0 + 4);
        const float4 b0 = *reinterpret_cast<const float4*>(a.beta + c0);
        const float4 b1 = *reinterpret_cast<const float4*>(a.beta + c0 + 4);
        const float gam[8] = {g0.x, g0.y, g0.z, g0.w, g1.x, g1.y, g1.z, g1.w};
        const float bet[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
        float x[8];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const float2 f = __half22float2(h[i]);
            x[2 * i] = f.x;
            x[2 * i + 1] = f.y;
        }
        uint4 o;
        __half2* oh = reinterpret_cast<__half2*>(&o);
#pragma unroll
        for (int i = 0; i < 8; i += 2) {
            const int ga = (c0 + i) / cpg, gb = (c0 + i + 1) / cpg;
            float y0 = (x[i] - s_mean[ga]) * s_rstd[ga] * gam[i] + bet[i];
            float y1 = (x[i + 1] - s_mean[gb]) * s_rstd[gb] * gam[i + 1] + bet[i + 1];
            if (a.silu) {
                y0 = silu_f(y0);
                y1 = silu_f(y1);
            }
            oh[i >> 1] = __floats2half2_rn(y0, y1);
        }
        *reinterpret_cast<uint4*>(a.y + ((long)b * a.hw + p) * a.ldy + c0) = o;
    }
}

// Single-launch variant: statistics, a per-batch-item grid barrier (cooperative launch guarantees co-residency),
// then normalise straight from the registers that still hold the chunk.  counters: 2 ints per batch item, zero
// between launches (the last CTA to leave re-arms them).
constexpr int GN_CACHE = 12;
__global__ void __launch_bounds__(512) gn_fused_kernel(GroupNormArgs a, int ppc, int vc, int rpi, int* counters) {
    B2_PDL_ENTRY();
    extern __shared__ float sm[];
    __shared__ float s_mean[64], s_rstd[64];
    const int C = a.ca + a.cb;
    const int chunk = blockIdx.x, b = blockIdx.y, nchunks = gridDim.x;
    const int col = threadIdx.x % vc, prow = threadIdx.x / vc;
    const int c0 = col * 8;
    const bool from_a = c0 < a.ca;
    const __half* base = from_a ? a.xa + c0 : a.xb + (c0 - a.ca);
    const int ld = from_a ? a.lda : a.ldb;
    const int p_begin = chunk * ppc, p_end = min(a.hw, p_begin + ppc);
    uint4 cache[GN_CACHE];
    float s[8], q[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) s[i] = q[i] = 0.f;
    if (prow < rpi) {
#pragma unroll
        for (int it = 0; it < GN_CACHE; ++it) {
            const int p = p_begin + prow + it * rpi;
            if (p < p_end) {
                const uint4 u = *reinterpret_cast<const uint4*>(base + ((long)b * a.hw + p) * ld);
                cache[it] = u;
                const __half2* h = reinterpret_cast<const __half2*>(&u);
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const float2 f = __half22float2(h[i]);
                    s[2 * i] += f.x; q[2 * i] += f.x * f.x;
                    s[2 * i + 1] += f.y; q[2 * i + 1] += f.y * f.y;
                }
            }
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            sm[((long)prow * C + c0 + i) * 2] = s[i];
            sm[((long)prow * C + c0 + i) * 2 + 1] = q[i];
        }
    }
    __syncthreads();
    const int cpg = C / a.groups;
    {
        // 8 lanes per group: lane `part` sums entries part, part+8, ... of the group's cpg*rpi (channel,row) pairs, then a
        // fixed 3-step shuffle tree combines the 8 parts
        const int part = threadIdx.x & 7;
        const int nent = cpg * rpi;
        for (int g = threadIdx.x >> 3; g < a.groups; g += blockDim.x >> 3) {
            float gs = 0.f, gq = 0.f;
            for (int e = part; e < nent; e += 8) {
                const int c = g * cpg + e % cpg, r = e / cpg;
                gs += sm[((long)r * C + c) * 2];
                gq += sm[((long)r * C + c) * 2 + 1];
            }
#pragma unroll
            for (int o = 4; o > 0; o >>= 1) {
                gs += __shfl_xor_sync(0xffffffffu, gs, o);
                gq += __shfl_xor_sync(0xffffffffu, gq, o);
            }
            if (part == 0)
                reinterpret_cast<float2*>(a.partial)[((long)b * a.groups + g) * GN_MAX_CHUNKS + chunk] = make_float2(gs, gq);
        }
    }
    // affine parameters: fetched now so their latency hides behind the grid barrier
    const float4 g0 = *reinterpret_cast<const float4*>(a.gamma + c0);
    const float4 g1 = *reinterpret_cast<const float4*>(a.gamma + c0 + 4);
    const float4 b0 = *reinterpret_cast<const float4*>(a.beta + c0);
    const float4 b1 = *reinterpret_cast<const float4*>(a.beta + c0 + 4);
    // ---- barrier over the CTAs of this batch item
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) {
        int* cnt = counters + 2 * b;
        atomicAdd(cnt, 1);
        const uint64_t t0 = globaltimer_ns_ew();
        while (true) {
            int seen;
            asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(seen) : "l"(cnt) : "memory");
            if (seen >= nchunks) break;
            __nanosleep(32);
            if (globaltimer_ns_ew() - t0 > 4000000000ull) {
                printf("b2: groupnorm grid barrier timeout\n");
                __trap();
            }
        }
        if (atomicAdd(cnt + 1, 1) == nchunks - 1) {  // last one out re-arms both counters for the next launch
            cnt[1] = 0;
            __threadfence();
            cnt[0] = 0;
        }
        __threadfence();
    }
    __syncthreads();
    gn_finalize_stats(a, b, nchunks, sm, s_mean, s_rstd);  // sm (>= 16*G*2 floats) is free again
    if (prow < rpi) {
        const float gam[8] = {g0.x, g0.y, g0.z, g0.w, g1.x, g1.y, g1.z, g1.w};
        const float bet[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
        float mu[8], rs[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int g = (c0 + i) / cpg;
            mu[i] = s_mean[g];
            rs[i] = s_rstd[g] * gam[i];
        }
#pragma unroll
        for (int it = 0; it < GN_CACHE; ++it) {
            const int p = p_begin + prow + it * rpi;
            if (p < p_end) {
                const __half2* h = reinterpret_cast<const __half2*>(&cache[it]);
                uint4 o;
                __half2* oh = reinterpret_cast<__half2*>(&o);
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const float2 f = __half22float2(h[i]);
                    float y0 = (f.x - mu[2 * i]) * rs[2 * i] + bet[2 * i];
                    float y1 = (f.y - mu[2 * i + 1]) * rs[2 * i + 1] + bet[2 * i + 1];
                    if (a.silu) {
                        y0 = silu_f(y0);
                        y1 = silu_f(y1);
                    }
                    oh[i] = __floats2half2_rn(y0, y1);
                }
                *reinterpret_cast<uint4*>(a.y + ((long)b * a.hw + p) * a.ldy + c0) = o;
            }
        }
    }
}

static thread_local int g_gn_last_launches = 0;
int groupnorm_last_launch_count() { return g_gn_last_launches; }
// ---- cluster variant (default when it fits): one thread-block cluster per (batch item, group).  The group's
// cpg = C/groups channels are a contiguous 2*cpg-byte run per pixel; the pixels are split over the 1/2/4/8 CTAs of the
// cluster, every thread keeps its <= 32 half2 words in registers, the (sum, sumsq) pairs of the CTAs are pushed into
// every peer's shared memory, one cluster barrier, then each CTA normalises straight from registers.  No grid barrier,
// no workspace, an ordinary (PDL-capable) launch: ~3x shorter than the cooperative whole-grid kernel at batch 1,
// where GroupNorm is pure latency (61 launches per SD-Turbo frame).
constexpr int GNC_THREADS = 240;   // a multiple of cpg/2 for cpg in {10, 20, 30, 40, 60, 80}: a thread owns one channel pair
constexpr int GNC_ITEMS = 32;
__global__ void __launch_bounds__(GNC_THREADS, 2) gn_cluster_kernel(GroupNormArgs a, int ppc) {
    __shared__ float2 part[8];   // (sum, sumsq) of every CTA of the cluster, pushed by its owner
    __shared__ float2 red[8];
    const int g = blockIdx.x, b = blockIdx.y, rank = blockIdx.z, nrank = gridDim.z;
    const int C = a.ca + a.cb, cpg = C / a.groups, wpp = cpg >> 1;
    const int t = threadIdx.x;
    const int wq = t % wpp, prow = t / wpp, pstep = GNC_THREADS / wpp;
    const int c = g * cpg + 2 * wq;
    const bool from_a = c < a.ca;
    const __half* src = from_a ? a.xa + c : a.xb + (c - a.ca);
    const int ld = from_a ? a.lda : a.ldb;
    const float2 gm = *reinterpret_cast<const float2*>(a.gamma + c);   // parameters: not produced by the previous kernel
    const float2 bt = *reinterpret_cast<const float2*>(a.beta + c);
    // A CTA may only touch a peer's shared memory once that peer is executing (compute-sanitizer racecheck: "block that might
    // not have entered yet"): every CTA arrives on the cluster barrier here and waits on it right before its DSMEM stores.
    if (nrank > 1) cluster_arrive_relaxed();
    B2_PDL_ENTRY();
    const int p0 = rank * ppc, p1 = min(a.hw, p0 + ppc);
    const long rowbase = (long)b * a.hw;
    uint32_t v[GNC_ITEMS];
#pragma unroll
    for (int k = 0; k < GNC_ITEMS; ++k) {
        const int p = p0 + prow + k * pstep;
        v[k] = 0u;
        if (p < p1) v[k] = *reinterpret_cast<const uint32_t*>(src + (rowbase + p) * ld);
    }
    float s = 0.f, q = 0.f;
#pragma unroll
    for (int k = 0; k < GNC_ITEMS; ++k) {   // out-of-range items are zero: they add nothing
        const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&v[k]));
        s += f.x + f.y;
        q += f.x * f.x + f.y * f.y;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        s += __shfl_xor_sync(0xffffffffu, s, o);
        q += __shfl_xor_sync(0xffffffffu, q, o);
    }
    if ((t & 31) == 0) red[t >> 5] = make_float2(s, q);
    __syncthreads();
    if (nrank > 1) cluster_wait();   // all peers have started (they arrived before their loads): remote stores are legal now
    if (t == 0) {
        float2 tot = make_float2(0.f, 0.f);
#pragma unroll
        for (int w = 0; w < (GNC_THREADS + 31) / 32; ++w) { tot.x += red[w].x; tot.y += red[w].y; }
        if (nrank == 1) part[0] = tot;
        else {
            const uint32_t slot = smem_u32(&part[rank]);
            for (int r = 0; r < nrank; ++r) dsmem_st_f2(dsmem_map(slot, (uint32_t)r), tot.x, tot.y);
        }
    }
    if (nrank > 1) cluster_sync_all();   // release/acquire over the cluster: every peer's pair has landed
    else __syncthreads();
    float S = 0.f, Q = 0.f;
    for (int r = 0; r < nrank; ++r) { S += part[r].x; Q += part[r].y; }   // fixed order => deterministic
    const float inv_n = 1.0f / ((float)a.hw * (float)cpg);
    const float mean = S * inv_n;
    const float rstd = rsqrtf(fmaxf(Q * inv_n - mean * mean, 0.f) + a.eps);
    const float ax = rstd * gm.x, ay = rstd * gm.y;
    const float bx = bt.x - mean * ax, by = bt.y - mean * ay;
    __half* dst = a.y + c;
#pragma unroll
    for (int k = 0; k < GNC_ITEMS; ++k) {
        const int p = p0 + prow + k * pstep;
        if (p < p1) {
            const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&v[k]));
            float y0 = f.x * ax + bx, y1 = f.y * ay + by;
            if (a.silu) {
                y0 = y0 / (1.0f + __expf(-y0));
                y1 = y1 / (1.0f + __expf(-y1));
            }
            *reinterpret_cast<__half2*>(dst + (rowbase + p) * a.ldy) = __floats2half2_rn(y0, y1);
        }
    }
}

// cluster size for gn_cluster_kernel, or 0 when the shape does not fit it
static int gn_cluster_size(const GroupNormArgs& a) {
    static const bool off = getenv("B2_NO_GN_CLUSTER") != nullptr;
    const int C = a.ca + a.cb;
    if (off || C % a.groups) return 0;
    const int cpg = C / a.groups;
    if ((cpg & 1) || (a.ca & 1) || GNC_THREADS % (cpg >> 1) != 0 || (a.lda & 1) || (a.cb && (a.ldb & 1)) || (a.ldy & 1)) return 0;
    const long words = (long)a.hw * (cpg >> 1);
    const long cap = (long)GNC_THREADS * GNC_ITEMS;
    static const char* mc = getenv("B2_GN_ITEMS");   // tuning: max half2 words per thread (default GNC_ITEMS)
    const int max_items = mc ? atoi(mc) : GNC_ITEMS;
    for (int cl = 1; cl <= 8; cl <<= 1) {
        const int ppc = (a.hw + cl - 1) / cl;
        const int pstep = GNC_THREADS / (cpg >> 1);
        if ((long)((ppc + pstep - 1) / pstep) <= max_items && words <= cap * cl) return cl;
    }
    return 0;
}

int groupnorm_plan(const GroupNormArgs& a, int* threads, int* pixels_per_cta) {
    const int cl = gn_cluster_size(a);
    if (threads) *threads = cl ? GNC_THREADS : 0;
    if (pixels_per_cta) *pixels_per_cta = cl ? (a.hw + cl - 1) / cl : 0;
    return cl;
}

size_t groupnorm_partial_floats(int nb, int groups) { return (size_t)nb * GN_MAX_CHUNKS * groups * 2 + 64; }

int groupnorm_launch(const GroupNormArgs& a, cudaStream_t s) {
    const int C = a.ca + a.cb;
    if (C % a.groups != 0 || a.groups > 64 || (C & 7) || (a.ca & 7) || (a.lda & 7) || (a.cb && (a.ldb & 7)) || (a.ldy & 7) ||
        !a.partial) {
        b2_set_error("groupnorm: unsupported channels %d+%d groups %d (need multiples of 8 and a workspace)", a.ca, a.cb,
                     a.groups);
        return -1;
    }
    if (const int cl = gn_cluster_size(a)) {
        const int ppc = (a.hw + cl - 1) / cl;
        B2_LAUNCHED("gn_cluster", launch_k(gn_cluster_kernel, dim3(a.groups, a.nb, cl), dim3(GNC_THREADS), 0, s, cl, a, ppc));
        g_gn_last_launches = 1;
        return 0;
    }
    const int vc = C / 8;
    if (vc > 512) {
        b2_set_error("groupnorm: %d channels exceed one CTA row", C);
        return -1;
    }
    int rpi = 512 / vc;            // pixel rows per iteration
    if (rpi > 8) rpi = 8;
    int ppc = (a.hw + GN_MAX_CHUNKS - 1) / GN_MAX_CHUNKS;
    if (ppc < 1) ppc = 1;
    if (rpi > ppc) rpi = ppc;
    const int nchunks = (a.hw + ppc - 1) / ppc;
    const int threads = ((vc * rpi + 31) / 32) * 32;
    size_t smem = (size_t)rpi * C * 2 * sizeof(float);
    if (smem < 16 * 64 * 2 * sizeof(float)) smem = 16 * 64 * 2 * sizeof(float);  // also the stats-finalise scratch
    static bool attr = false;
    if (!attr) {
        cudaFuncSetAttribute(gn_stats_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024);
        cudaFuncSetAttribute(gn_fused_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024);
        attr = true;
    }
    // single cooperative launch when the whole grid is co-resident and a chunk fits the register cache
    int per_sm = 0;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, gn_fused_kernel, threads, smem);
    const bool fits = (ppc + rpi - 1) / rpi <= GN_CACHE && (long)nchunks * a.nb <= (long)per_sm * 148 && a.nb <= 16;
    if (fits && a.counters) {
        cudaLaunchConfig_t cfg{};
        cfg.gridDim = dim3(nchunks, a.nb);
        cfg.blockDim = dim3(threads);
        cfg.dynamicSmemBytes = smem;
        cfg.stream = s;
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeCooperative;
        at[0].val.cooperative = 1;
        cfg.attrs = at;
        cfg.numAttrs = 1;
        cudaError_t e = cudaLaunchKernelEx(&cfg, gn_fused_kernel, a, ppc, vc, rpi, a.counters);
        if (e != cudaSuccess) {
            b2_set_error("gn_fused launch: %s", cudaGetErrorString(e));
            return -1;
        }
        g_gn_last_launches = 1;
        return 0;
    }
    B2_LAUNCHED("gn_stats", launch_k(gn_stats_kernel, dim3(nchunks, a.nb), dim3(threads), smem, s, 1, a, ppc, vc, rpi));
    const long vec_per_batch = (long)a.hw * vc;
    long blocks = (vec_per_batch + 255) / 256;
    const long cap = (148 * 4 + a.nb - 1) / a.nb;
    if (blocks > cap) blocks = cap;
    B2_LAUNCHED("gn_apply", launch_k(gn_apply_kernel, dim3((unsigned)blocks, a.nb), dim3(256), 0, s, 1, a, nchunks, vec_per_batch));
    g_gn_last_launches = 2;
    return 0;
}

// ------------------------------------------------------------------------------------------ LayerNorm
// One warp per row; the row (<= 5 x 16 B per lane, C <= 1280) stays in registers between the statistics and the
// normalisation, and gamma/beta (parameters, not produced by the previous kernel) are fetched before the PDL wait.
constexpr int LN_MAXK = 5;
__global__ void __launch_bounds__(256) layernorm_kernel(const __half* __restrict__ x, int ldx, const float* __restrict__ gamma,
                                                        const float* __restrict__ beta, __half* __restrict__ y, int ldy, long rows,
                                                        int c, float eps) {
    const long row = (long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    const int chunks = c >> 3;
    float4 g[LN_MAXK][2], bt[LN_MAXK][2];
#pragma unroll
    for (int k = 0; k < LN_MAXK; ++k) {
        const int ch = lane + 32 * k;
        if (ch < chunks) {
            g[k][0] = __ldg(reinterpret_cast<const float4*>(gamma) + 2 * ch);
            g[k][1] = __ldg(reinterpret_cast<const float4*>(gamma) + 2 * ch + 1);
            bt[k][0] = __ldg(reinterpret_cast<const float4*>(beta) + 2 * ch);
            bt[k][1] = __ldg(reinterpret_cast<const float4*>(beta) + 2 * ch + 1);
        }
    }
    B2_PDL_ENTRY();
    if (row >= rows) return;
    const __half* xr = x + row * ldx;
    uint4 xv[LN_MAXK];
#pragma unroll
    for (int k = 0; k < LN_MAXK; ++k) {
        const int ch = lane + 32 * k;
        xv[k] = make_uint4(0, 0, 0, 0);
        if (ch < chunks) xv[k] = reinterpret_cast<const uint4*>(xr)[ch];
    }
    float s = 0.f, ss = 0.f;
#pragma unroll
    for (int k = 0; k < LN_MAXK; ++k) {   // absent chunks are zero: they add nothing
        const __half2* h = reinterpret_cast<const __half2*>(&xv[k]);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const float2 f = __half22float2(h[i]);
            s += f.x + f.y;
            ss += f.x * f.x + f.y * f.y;
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        s += __shfl_xor_sync(0xffffffffu, s, o);
        ss += __shfl_xor_sync(0xffffffffu, ss, o);
    }
    const float mean = s / c;
    const float rstd = rsqrtf(fmaxf(ss / c - mean * mean, 0.f) + eps);
    __half* yr = y + row * ldy;
#pragma unroll
    for (int k = 0; k < LN_MAXK; ++k) {
        const int ch = lane + 32 * k;
        if (ch < chunks) {
            const __half2* h = reinterpret_cast<const __half2*>(&xv[k]);
            const float* gp = reinterpret_cast<const float*>(&g[k][0]);
            const float* bp = reinterpret_cast<const float*>(&bt[k][0]);
            uint4 o;
            __half2* oh = reinterpret_cast<__half2*>(&o);
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const float2 f = __half22float2(h[i]);
                oh[i] = __floats2half2_rn((f.x - mean) * rstd * gp[2 * i] + bp[2 * i], (f.y - mean) * rstd * gp[2 * i + 1] + bp[2 * i + 1]);
            }
            reinterpret_cast<uint4*>(yr)[ch] = o;
        }
    }
}

int layernorm_launch(const __half* x, int ldx, const float* gamma, const float* beta, __half* y, int ldy,
                     long rows, int c, float eps, cudaStream_t s) {
    if ((c & 7) || (ldx & 7) || (ldy & 7) || c > LN_MAXK * 256 || (reinterpret_cast<uintptr_t>(gamma) & 15) || (reinterpret_cast<uintptr_t>(beta) & 15)) {
        b2_set_error("layernorm: c/ld must be multiples of 8, c <= %d, gamma/beta 16-byte aligned (c=%d)", LN_MAXK * 256, c);
        return -1;
    }
    const int wpb = 8;
    B2_LAUNCHED("layernorm", launch_k(layernorm_kernel, dim3((unsigned)((rows + wpb - 1) / wpb)), dim3(wpb * 32), 0, s, 1, x, ldx, gamma,
                                      beta, y, ldy, rows, c, eps));
    return 0;
}

// ------------------------------------------------------------------------------------------ upsample
__global__ void upsample2x_kernel(const uint4* __restrict__ x, uint4* __restrict__ y, int nb, int h, int w, int c8) {
    B2_PDL_ENTRY();
    const long total = (long)nb * (2 * h) * (2 * w) * c8;
    for (long e = (long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long)gridDim.x * blockDim.x) {
        const int cc = (int)(e % c8);
        long p = e / c8;
        const int wo = (int)(p % (2 * w));
        p /= (2 * w);
        const int ho = (int)(p % (2 * h));
        const int n = (int)(p / (2 * h));
        y[e] = x[(((long)n * h + (ho >> 1)) * w + (wo >> 1)) * c8 + cc];
    }
}

int upsample2x_launch(const __half* x, __half* y, int nb, int h, int w, int c, cudaStream_t s) {
    if (c & 7) {
        b2_set_error("upsample2x: c %% 8 != 0");
        return -1;
    }
    const long total = (long)nb * 4 * h * w * (c / 8);
    const int threads = 256;
    long blocks = (total + threads - 1) / threads;
    if (blocks > 148 * 16) blocks = 148 * 16;
    B2_LAUNCHED("upsample2x", launch_k(upsample2x_kernel, dim3((unsigned)blocks), dim3(threads), 0, s, 1,
                                       reinterpret_cast<const uint4*>(x), reinterpret_cast<uint4*>(y), nb, h, w, c / 8));
    return 0;
}

// ------------------------------------------------------------------------------------------ small conv
// thread = (pixel, 64 output channels): the 3x3xCIN patch lives in registers, the fp32 weights [k][cout]
// (k = tap*CIN + c, prepared once by smallconv_prep_launch) in shared memory where a warp reads them as broadcasts.
__global__ void smallconv_prep_kernel(const __half* __restrict__ w_oihw, float* __restrict__ wt, int cout, int cin) {
    const int K = cin * 9;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < K * cout; i += gridDim.x * blockDim.x) {
        const int o = i % cout, k = i / cout;
        const int tap = k / cin, c = k % cin;
        wt[i] = __half2float(w_oihw[((long)o * cin + c) * 9 + tap]);
    }
}
int smallconv_prep_launch(const __half* w_oihw, float* wt, int cout, int cin, cudaStream_t s) {
    smallconv_prep_kernel<<<(cin * 9 * cout + 255) / 256, 256, 0, s>>>(w_oihw, wt, cout, cin);
    B2_CHECK_LAUNCH("smallconv_prep");
    return 0;
}

template <int CIN>
__global__ void __launch_bounds__(128) smallconv_kernel(SmallConvArgs a, int G) {
    B2_PDL_ENTRY();
    extern __shared__ float ws[];  // [CIN*9][G] weights of this CTA's G-channel output group, then bias[G]
    constexpr int K = CIN * 9;
    const int cout = a.cout;
    const int cg = blockIdx.y;   // G-channel output group (G = 64, or 16 for small images: more CTAs)
    const int gq = G >> 2;
    for (int i = threadIdx.x; i < K * gq; i += blockDim.x) {
        const int k = i / gq, j = i - k * gq;
        reinterpret_cast<float4*>(ws)[i] = *reinterpret_cast<const float4*>(a.wt + (long)k * cout + cg * G + 4 * j);
    }
    float* bs = ws + K * G;
    for (int i = threadIdx.x; i < G; i += blockDim.x) bs[i] = a.bias ? a.bias[cg * G + i] : 0.f;
    __syncthreads();
    const int npix = a.nb * a.h * a.w_;           // < 2^31 (checked by the launcher)
    const bool same_size = a.in_h == a.h && a.in_w == a.w_;   // no resize: skip the per-tap integer divisions
    for (int p = blockIdx.x * blockDim.x + threadIdx.x; p < npix; p += gridDim.x * blockDim.x) {
        const int xw = p % a.w_;
        const int yh = (p / a.w_) % a.h;
        const int n_out = p / (a.w_ * a.h);
        const int n = n_out < a.uc_rows ? n_out : n_out - a.uc_rows;   // source batch row
        float patch[K];
#pragma unroll
        for (int tap = 0; tap < 9; ++tap) {
            const int yy = yh + tap / 3 - 1, xx = xw + tap % 3 - 1;
            const bool in = (yy >= 0) && (yy < a.h) && (xx >= 0) && (xx < a.w_);
            // nearest resize (VaeImageProcessor.resize -> F.interpolate default mode): src = floor(dst*in/out)
            int sy = 0, sx = 0;
            if (in) {
                if (same_size) { sy = yy; sx = xx; }
                else { sy = (int)(((long)yy * a.in_h) / a.h); sx = (int)(((long)xx * a.in_w) / a.w_); }
            }
            const long base = (((long)n * a.in_h + sy) * a.in_w + sx) * CIN;
#pragma unroll
            for (int c = 0; c < CIN; ++c) {
                float v = 0.f;
                if (in) {
                    if (a.flags & (SC_IN_F32_NCHW | SC_IN_F16_NCHW)) {
                        // lib/pipeline.py:65 hands StreamDiffusion a (3,H,W) float tensor in [0,1]
                        const long idx = (((long)n * CIN + c) * a.in_h + sy) * a.in_w + sx;
                        v = (a.flags & SC_IN_F32_NCHW) ? reinterpret_cast<const float*>(a.x)[idx]
                                                       : __half2float(reinterpret_cast<const __half*>(a.x)[idx]);
                    } else if (a.flags & SC_IN_U8) {
                        // lib/pipeline.py:61 convertto(scale=1/255); the 2x-1 of VaeImageProcessor and the
                        // (x+1)/2 of EncoderTiny cancel
                        v = (float)reinterpret_cast<const uint8_t*>(a.x)[base + c] * (1.0f / 255.0f);
                    } else {
                        v = __half2float(reinterpret_cast<const __half*>(a.x)[base + c]);
                        if (a.flags & SC_IN_TANH3) v = tanhf(v * (1.0f / 3.0f)) * 3.0f;
                    }
                    // operands of the reference engines are fp16
                    v = __half2float(__float2half_rn(v));
                }
                patch[tap * CIN + c] = v;
            }
        }
        // 16 output channels per pass: the patch stays in registers, the accumulators are reused (64 at once needed
        // ~240 registers per thread => 2 CTAs per SM and a latency-bound FMA stream)
        __half* dst = a.y + (long)p * a.ldy + cg * G;
#pragma unroll 1
        for (int q = 0; q < G; q += 16) {
            float acc[16];
#pragma unroll
            for (int o = 0; o < 16; ++o) acc[o] = bs[q + o];
#pragma unroll
            for (int k = 0; k < K; ++k) {
                const float v = patch[k];
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const float4 w4 = *reinterpret_cast<const float4*>(ws + k * G + q + 4 * j);
                    acc[4 * j] += v * w4.x; acc[4 * j + 1] += v * w4.y; acc[4 * j + 2] += v * w4.z; acc[4 * j + 3] += v * w4.w;
                }
            }
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                uint4 u;
                __half2* hh = reinterpret_cast<__half2*>(&u);
#pragma unroll
                for (int o = 0; o < 4; ++o) {
                    float v0 = acc[8 * j + 2 * o], v1 = acc[8 * j + 2 * o + 1];
                    if (a.flags & SC_OUT_RELU) {
                        v0 = fmaxf(v0, 0.f);
                        v1 = fmaxf(v1, 0.f);
                    }
                    hh[o] = __floats2half2_rn(v0, v1);
                }
                reinterpret_cast<uint4*>(dst + q)[j] = u;
            }
        }
    }
}

int smallconv_launch(const SmallConvArgs& a, cudaStream_t s) {
    if ((a.cout & 63) || (a.ldy & 7) || (a.cin != 3 && a.cin != 4) || !a.wt) {
        b2_set_error("smallconv: cin %d cout %d unsupported (cout must be a multiple of 64; prepared weights required)", a.cin, a.cout);
        return -1;
    }
    const long npix = (long)a.nb * a.h * a.w_;
    if (npix >= (1l << 31) - 128 * 148 * 32) {
        b2_set_error("smallconv: %ld pixels exceed the 32-bit index range", npix);
        return -1;
    }
    long blocks = (npix + 127) / 128;
    const int G = blocks * (a.cout / 64) < 148 * 4 ? 16 : 64;   // few pixels: narrower channel groups, more CTAs
    const size_t smem = ((size_t)a.cin * 9 * G + G) * sizeof(float);
    const int groups = a.cout / G;
    const long cap = (148 * 16 + groups - 1) / groups;   // two full waves of 8 CTAs per SM; beyond that, grid-stride
    if (blocks > cap) blocks = cap;
    static bool attr = false;
    if (!attr) {
        cudaFuncSetAttribute(smallconv_kernel<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024);
        cudaFuncSetAttribute(smallconv_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024);
        attr = true;
    }
    if (a.cin == 3) B2_LAUNCHED("smallconv", launch_k(smallconv_kernel<3>, dim3((unsigned)blocks, groups), dim3(128), smem, s, 1, a, G));
    else B2_LAUNCHED("smallconv", launch_k(smallconv_kernel<4>, dim3((unsigned)blocks, groups), dim3(128), smem, s, 1, a, G));
    return 0;
}

// ------------------------------------------------------------------------------------------ LCM step
__global__ void lcm_step_kernel(__half* __restrict__ x, const __half* __restrict__ eps,
                                const __half* __restrict__ noise, const float* __restrict__ coef,
                                __half* __restrict__ out_latent, int T, int hw, int do_add_noise) {
    B2_PDL_ENTRY();
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= hw) return;
    const float* alpha = coef;
    const float* beta = coef + T;
    const float* c_skip = coef + 2 * T;
    const float* c_out = coef + 3 * T;
    float prev[4] = {0.f, 0.f, 0.f, 0.f};
    for (int i = 0; i < T; ++i) {
        const long off = ((long)i * hw + p) * 4;
        const uint2 ux = *reinterpret_cast<const uint2*>(x + off);
        const uint2 ue = *reinterpret_cast<const uint2*>(eps + off);
        const __half2* hx = reinterpret_cast<const __half2*>(&ux);
        const __half2* he = reinterpret_cast<const __half2*>(&ue);
        float xv[4], ev[4], x0[4];
        *reinterpret_cast<float2*>(&xv[0]) = __half22float2(hx[0]);
        *reinterpret_cast<float2*>(&xv[2]) = __half22float2(hx[1]);
        *reinterpret_cast<float2*>(&ev[0]) = __half22float2(he[0]);
        *reinterpret_cast<float2*>(&ev[2]) = __half22float2(he[1]);
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            const float f = (xv[c] - beta[i] * ev[c]) / alpha[i];
            x0[c] = c_out[i] * f + c_skip[i] * xv[c];
        }
        if (i > 0) {
            // slot i of the next call = re-noised x0 of slot i-1 (computed last iteration)
            float nv[4] = {0.f, 0.f, 0.f, 0.f};
            if (do_add_noise) {
                const uint2 un = *reinterpret_cast<const uint2*>(noise + off);
                const __half2* hn = reinterpret_cast<const __half2*>(&un);
                *reinterpret_cast<float2*>(&nv[0]) = __half22float2(hn[0]);
                *reinterpret_cast<float2*>(&nv[2]) = __half22float2(hn[1]);
            }
            uint2 uo;
            __half2* ho = reinterpret_cast<__half2*>(&uo);
            ho[0] = __floats2half2_rn(alpha[i] * prev[0] + beta[i] * nv[0], alpha[i] * prev[1] + beta[i] * nv[1]);
            ho[1] = __floats2half2_rn(alpha[i] * prev[2] + beta[i] * nv[2], alpha[i] * prev[3] + beta[i] * nv[3]);
            *reinterpret_cast<uint2*>(x + off) = uo;
        }
#pragma unroll
        for (int c = 0; c < 4; ++c) prev[c] = x0[c];
    }
    uint2 uo;
    __half2* ho = reinterpret_cast<__half2*>(&uo);
    ho[0] = __floats2half2_rn(prev[0], prev[1]);
    ho[1] = __floats2half2_rn(prev[2], prev[3]);
    *reinterpret_cast<uint2*>(out_latent + (long)p * 4) = uo;
}

int lcm_step_launch(__half* x, const __half* eps, const __half* noise, const float* coef, __half* out_latent,
                    int T, int hw, int do_add_noise, cudaStream_t s) {
    B2_LAUNCHED("lcm_step", launch_k(lcm_step_kernel, dim3((hw + 127) / 128), dim3(128), 0, s, 1, x, eps, noise, coef, out_latent, T, hw,
                                     do_add_noise));
    return 0;
}

// ------------------------------------------------------------------------------------------ LCM step with residual CFG
__device__ __forceinline__ void ld4h(const __half* p, float v[4]) {
    const uint2 u = *reinterpret_cast<const uint2*>(p);
    const __half2* h = reinterpret_cast<const __half2*>(&u);
    *reinterpret_cast<float2*>(&v[0]) = __half22float2(h[0]);
    *reinterpret_cast<float2*>(&v[2]) = __half22float2(h[1]);
}
__device__ __forceinline__ void st4h(__half* p, const float v[4]) {
    uint2 u;
    __half2* h = reinterpret_cast<__half2*>(&u);
    h[0] = __floats2half2_rn(v[0], v[1]);
    h[1] = __floats2half2_rn(v[2], v[3]);
    *reinterpret_cast<uint2*>(p) = u;
}

// One thread per latent pixel walks the T slots in order, so the stock-noise shift (slot i reads slot i-1's old value) and
// the latent-buffer re-noise (slot i gets slot i-1's x0) need no second pass.  eps rows: [uncond rows (u) | text rows (T)].
__global__ void lcm_cfg_step_kernel(__half* __restrict__ x, const __half* __restrict__ eps, const __half* __restrict__ noise,
                                    __half* __restrict__ stock, const float* __restrict__ coef, __half* __restrict__ out_latent,
                                    int T, int hw, int do_add_noise, int cfg_type, float guidance, float delta) {
    B2_PDL_ENTRY();
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= hw) return;
    const float* alpha = coef;
    const float* beta = coef + T;
    const float* c_skip = coef + 2 * T;
    const float* c_out = coef + 3 * T;
    const bool full = cfg_type == CFG_FULL;
    const bool residual = cfg_type == CFG_SELF || cfg_type == CFG_INITIALIZE;   // eps_uncond = delta * stock noise
    const int u = cfg_type == CFG_INITIALIZE ? 1 : (full ? T : 0);
    float n0[4], prev_x0[4] = {0.f, 0.f, 0.f, 0.f}, prev_stock[4];
    ld4h(noise + (long)p * 4, n0);
    for (int i = 0; i < T; ++i) {
        const long off = ((long)i * hw + p) * 4;
        float xv[4], et[4], so[4], sv[4], eu[4], x0[4];
        ld4h(x + off, xv);
        ld4h(eps + off + (long)u * hw * 4, et);
        ld4h(stock + off, so);
        // predict_x0_batch (T > 1): stock = cat(init_noise[0:1], stock[:-1]);  initialize: stock[0] = eps of the uncond row
#pragma unroll
        for (int c = 0; c < 4; ++c) sv[c] = T > 1 ? (i == 0 ? n0[c] : prev_stock[c]) : so[c];
        if (cfg_type == CFG_INITIALIZE && i == 0) ld4h(eps + (long)p * 4, sv);
        if (full) ld4h(eps + off, eu);
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            if (!full) eu[c] = delta * sv[c];
            const float pred = eu[c] + guidance * (et[c] - eu[c]);
            x0[c] = c_out[i] * ((xv[c] - beta[i] * pred) / alpha[i]) + c_skip[i] * xv[c];
            if (residual) {
                // delta_x = scheduler_step(pred, beta * stock) * alpha_next / beta_next;  stock' = roll(init_noise, -1) + delta_x
                const float sc = beta[i] * sv[c];
                const float dx = c_out[i] * ((sc - beta[i] * pred) / alpha[i]) + c_skip[i] * sc;
                const float an = i + 1 < T ? alpha[i + 1] : 1.f, bn = i + 1 < T ? beta[i + 1] : 1.f;
                eu[c] = an * dx / bn;   // reuse: delta_x
            }
        }
        if (residual) {
            float nn[4];
            if (i + 1 < T) ld4h(noise + off + (long)hw * 4, nn);
            else { nn[0] = n0[0]; nn[1] = n0[1]; nn[2] = n0[2]; nn[3] = n0[3]; }
#pragma unroll
            for (int c = 0; c < 4; ++c) sv[c] = nn[c] + eu[c];
        }
        st4h(stock + off, sv);   // full: only the shift (the value never feeds the output)
        if (i > 0) {
            float nv[4] = {0.f, 0.f, 0.f, 0.f}, o[4];
            if (do_add_noise) ld4h(noise + off, nv);
#pragma unroll
            for (int c = 0; c < 4; ++c) o[c] = alpha[i] * prev_x0[c] + beta[i] * nv[c];
            st4h(x + off, o);
        }
#pragma unroll
        for (int c = 0; c < 4; ++c) { prev_x0[c] = x0[c]; prev_stock[c] = so[c]; }
    }
    st4h(out_latent + (long)p * 4, prev_x0);
}

int lcm_cfg_step_launch(__half* x, const __half* eps, const __half* noise, __half* stock, const float* coef, __half* out_latent,
                        int T, int hw, int do_add_noise, int cfg_type, float guidance, float delta, cudaStream_t s) {
    if (cfg_type != CFG_SELF && cfg_type != CFG_INITIALIZE && cfg_type != CFG_FULL) {
        b2_set_error("lcm_cfg_step: cfg_type %d is not self / initialize / full", cfg_type);
        return -1;
    }
    B2_LAUNCHED("lcm_cfg_step", launch_k(lcm_cfg_step_kernel, dim3((hw + 127) / 128), dim3(128), 0, s, 1, x, eps, noise, stock, coef,
                                         out_latent, T, hw, do_add_noise, cfg_type, guidance, delta));
    return 0;
}

// ------------------------------------------------------------------------------------------ post
__global__ void post_u8_kernel(const __half* __restrict__ y, int ldy, uint8_t* __restrict__ out, int nb, int h, int w) {
    B2_PDL_ENTRY();
    const long hw = (long)h * w;
    const long total = (long)nb * hw;
    const long p = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= total) return;
    const int n = (int)(p / hw);
    const long q = p % hw;
    const __half one = __float2half(1.0f), half_ = __float2half(0.5f), two = __float2half(2.0f);
    const __half zero = __float2half(0.0f), s255 = __float2half(255.0f);
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        __half v = y[p * ldy + c];
        v = __hsub(__hmul(v, two), one);        // DecoderTiny.forward: x.mul(2).sub(1)
        v = __hadd(__hmul(v, half_), half_);    // postprocess_image: x / 2 + 0.5
        v = __hmax(zero, __hmin(v, one));       // .clamp(0, 1)
        v = __hmul(v, s255);                    // lib/pipeline.py:74  frame * 255.0
        v = __hmax(zero, __hmin(v, s255));      // .clamp(0, 255)
        out[((long)n * 3 + c) * hw + q] = (uint8_t)__half2int_rz(v);  // .to(uint8): truncation
    }
}

__global__ void post_f16_kernel(const __half* __restrict__ y, int ldy, __half* __restrict__ out, int nb, int h, int w) {
    B2_PDL_ENTRY();
    const long hw = (long)h * w;
    const long p = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= (long)nb * hw) return;
    const int n = (int)(p / hw);
    const long q = p % hw;
#pragma unroll
    for (int c = 0; c < 3; ++c)
        out[((long)n * 3 + c) * hw + q] = __hsub(__hmul(y[p * ldy + c], __float2half(2.0f)), __float2half(1.0f));
}

int post_f16_launch(const __half* y_nhwc, int ldy, __half* out_nchw, int nb, int h, int w, cudaStream_t s) {
    const long total = (long)nb * h * w;
    B2_LAUNCHED("post_f16", launch_k(post_f16_kernel, dim3((unsigned)((total + 255) / 256)), dim3(256), 0, s, 1, y_nhwc, ldy, out_nchw, nb, h, w));
    return 0;
}

int post_u8_launch(const __half* y_nhwc, int ldy, uint8_t* out_nchw, int nb, int h, int w, cudaStream_t s) {
    const long total = (long)nb * h * w;
    B2_LAUNCHED("post_u8", launch_k(post_u8_kernel, dim3((unsigned)((total + 255) / 256)), dim3(256), 0, s, 1, y_nhwc, ldy, out_nchw, nb, h, w));
    return 0;
}

// ------------------------------------------------------------------------------------------ prepare-time
__global__ void small_linear_kernel(const float* __restrict__ in, int in_ld, const __half* __restrict__ w,
                                    const float* __restrict__ bias, float* __restrict__ out, int out_ld, int nb,
                                    int n, int k, int silu_in) {
    const long warp = ((long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (warp >= (long)nb * n) return;
    const int b = (int)(warp / n), j = (int)(warp % n);
    float acc = 0.f;
    for (int i = lane; i < k; i += 32) {
        float v = in[(long)b * in_ld + i];
        if (silu_in) v = v / (1.0f + expf(-v));
        acc += v * __half2float(w[(long)j * k + i]);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (lane == 0) out[(long)b * out_ld + j] = acc + (bias ? bias[j] : 0.f);
}

int small_linear_launch(const float* in, int in_ld, const __half* w, const float* bias, float* out, int out_ld,
                        int nb, int n, int k, int silu_in, cudaStream_t s) {
    const long warps = (long)nb * n;
    small_linear_kernel<<<(unsigned)((warps * 32 + 255) / 256), 256, 0, s>>>(in, in_ld, w, bias, out, out_ld, nb, n, k, silu_in);
    B2_CHECK_LAUNCH("small_linear");
    return 0;
}

__global__ void timestep_embedding_kernel(const float* __restrict__ t, float* __restrict__ out, int nb, int dim) {
    const int half_dim = dim / 2;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nb * half_dim) return;
    const int b = i / half_dim, j = i % half_dim;
    const float freq = expf(-logf(10000.0f) * (float)j / (float)half_dim);
    const float arg = t[b] * freq;
    out[(long)b * dim + j] = cosf(arg);             // flip_sin_to_cos=True: [cos | sin]
    out[(long)b * dim + half_dim + j] = sinf(arg);
}

int timestep_embedding_launch(const float* t, float* out, int nb, int dim, cudaStream_t s) {
    const int total = nb * (dim / 2);
    timestep_embedding_kernel<<<(total + 127) / 128, 128, 0, s>>>(t, out, nb, dim);
    B2_CHECK_LAUNCH("timestep_embedding");
    return 0;
}

__global__ void cast_f32_f16_kernel(const float* __restrict__ x, __half* __restrict__ y, long n) {
    for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x)
        y[i] = __float2half_rn(x[i]);
}
__global__ void cast_f16_f32_kernel(const __half* __restrict__ x, float* __restrict__ y, long n) {
    for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x)
        y[i] = __half2float(x[i]);
}
static unsigned grid_for(long n) {
    long b = (n + 255) / 256;
    if (b > 148 * 32) b = 148 * 32;
    if (b < 1) b = 1;
    return (unsigned)b;
}
int cast_f32_to_f16_launch(const float* x, __half* y, long n, cudaStream_t s) {
    cast_f32_f16_kernel<<<grid_for(n), 256, 0, s>>>(x, y, n);
    B2_CHECK_LAUNCH("cast_f32_f16");
    return 0;
}
int cast_f16_to_f32_launch(const __half* x, float* y, long n, cudaStream_t s) {
    cast_f16_f32_kernel<<<grid_for(n), 256, 0, s>>>(x, y, n);
    B2_CHECK_LAUNCH("cast_f16_f32");
    return 0;
}

__global__ void pack_conv_weight_kernel(const __half* __restrict__ w, __half* __restrict__ dst, int dst_ld, int koff,
                                        int o, int i, int taps, int c0, int cn) {
    const long total = (long)o * taps * cn;
    for (long e = (long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long)gridDim.x * blockDim.x) {
        const int c = (int)(e % cn);
        const int tap = (int)((e / cn) % taps);
        const int oo = (int)(e / ((long)cn * taps));
        dst[(long)oo * dst_ld + koff + tap * cn + c] = w[((long)oo * i + (c0 + c)) * taps + tap];
    }
}
int pack_conv_weight_launch(const __half* w_oihw, __half* dst, int dst_ld, int koff, int o, int i, int taps, int c0,
                            int cn, cudaStream_t s) {
    pack_conv_weight_kernel<<<grid_for((long)o * taps * cn), 256, 0, s>>>(w_oihw, dst, dst_ld, koff, o, i, taps, c0, cn);
    B2_CHECK_LAUNCH("pack_conv_weight");
    return 0;
}

__global__ void gather_rows_kernel(const __half* __restrict__ src, int src_ld, const int* __restrict__ perm,
                                   __half* __restrict__ dst, int dst_ld, int rows, int cols) {
    const long total = (long)rows * cols;
    for (long e = (long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long)gridDim.x * blockDim.x) {
        const int c = (int)(e % cols);
        const int r = (int)(e / cols);
        const int sr = perm ? perm[r] : r;
        dst[(long)r * dst_ld + c] = sr >= 0 ? src[(long)sr * src_ld + c] : __float2half(0.f);
    }
}
int gather_rows_launch(const __half* src, int src_ld, const int* perm, __half* dst, int dst_ld, int rows, int cols,
                       cudaStream_t s) {
    gather_rows_kernel<<<grid_for((long)rows * cols), 256, 0, s>>>(src, src_ld, perm, dst, dst_ld, rows, cols);
    B2_CHECK_LAUNCH("gather_rows");
    return 0;
}

// ---- LayerNorm folded into the consumer GEMM (load-time preparation; one warp per weight row) -----------------------
__global__ void scale_cols_kernel(__half* w, long rows, int k, const float* __restrict__ g) {
    const long r = (long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (r >= rows) return;
    for (int c = threadIdx.x & 31; c < k; c += 32) w[r * k + c] = __float2half_rn(__half2float(w[r * k + c]) * g[c]);
}
__global__ void row_sum_kernel(const __half* __restrict__ w, long rows, int k, float* out) {
    const long r = (long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (r >= rows) return;
    float a = 0.f;
    for (int c = threadIdx.x & 31; c < k; c += 32) a += __half2float(w[r * k + c]);
    for (int o = 16; o; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
    if ((threadIdx.x & 31) == 0) out[r] = a;
}
__global__ void row_dot_kernel(const __half* __restrict__ w, long rows, int k, const float* __restrict__ v,
                               const float* __restrict__ bias, float* out) {
    const long r = (long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (r >= rows) return;
    float a = 0.f;
    for (int c = threadIdx.x & 31; c < k; c += 32) a += __half2float(w[r * k + c]) * v[c];
    for (int o = 16; o; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
    if ((threadIdx.x & 31) == 0) out[r] = a + (bias ? bias[r] : 0.f);
}
int scale_cols_launch(__half* w, long rows, int k, const float* gamma, cudaStream_t s) {
    scale_cols_kernel<<<(unsigned)((rows + 7) / 8), 256, 0, s>>>(w, rows, k, gamma);
    B2_CHECK_LAUNCH("scale_cols");
    return 0;
}
int row_sum_launch(const __half* w, long rows, int k, float* out, cudaStream_t s) {
    row_sum_kernel<<<(unsigned)((rows + 7) / 8), 256, 0, s>>>(w, rows, k, out);
    B2_CHECK_LAUNCH("row_sum");
    return 0;
}
int row_dot_launch(const __half* w, long rows, int k, const float* v, const float* bias, float* out, cudaStream_t s) {
    row_dot_kernel<<<(unsigned)((rows + 7) / 8), 256, 0, s>>>(w, rows, k, v, bias, out);
    B2_CHECK_LAUNCH("row_dot");
    return 0;
}

}  // namespace b2
