// Fused train-mode BatchNorm2d + LeakyReLU(0.01) + Dropout(p) for the channels-last bf16 path:
// the "BN -> LeakyReLU -> Dropout" run between the two convolutions of every ConvBlock
// (utilities/UAPS_unet.py:37-43; batch statistics, eps 1e-5, momentum 0.1).
//
// The reference runs batch_norm (stats + transform), leaky_relu and dropout as separate ATen kernels,
// forward and backward: ten HBM round trips per block.  Here:
//   forward : bn_stats (read y) -> bn_act (read y, write a)                       2 + 4 B/element (bf16)
//   backward: bn_act_bwd_reduce (read g, y) -> bn_act_bwd (read g, y, write dy)   4 + 6 B/element
// The LeakyReLU sign and the dropout mask are recomputed in the backward pass from the saved conv
// output y and a Philox counter, so neither the activation nor a mask is stored.
//
// Layout: y is [npix, C] bf16, C a power of two in 8..256.  G = C/8 adjacent threads own the eight
// 16-byte chunks of a pixel; a thread's channels are fixed over its grid-stride loop, so per-channel
// sums are private registers until one shared-memory + one fp64 global atomic per channel per CTA.
#include <cstdlib>
#include <cooperative_groups.h>
#include <cuda_bf16.h>
#include "common.cuh"

namespace uaps {
namespace {

constexpr int BT = 256;
constexpr uint32_t kStreamBnDrop = 21;

__device__ __forceinline__ void unpack8(const uint4& r, float (&v)[8]) {
    const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&r);
#pragma unroll
    for (int i = 0; i < 4; ++i) { const float2 f = __bfloat1622float2(h[i]); v[2 * i] = f.x; v[2 * i + 1] = f.y; }
}
__device__ __forceinline__ uint4 pack8(const float (&v)[8]) {
    uint4 r;
    __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(&r);
#pragma unroll
    for (int i = 0; i < 4; ++i) h[i] = __floats2bfloat162_rn(v[2 * i], v[2 * i + 1]);
    return r;
}
__device__ __forceinline__ void keep8(uint64_t seed, uint64_t idx, float p, float (&k)[8]) {
    uint32_t r[4];
    Philox::draw4(seed, idx, kStreamBnDrop, r);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        k[2 * i] = ((float)(r[i] & 0xffffu) * (1.0f / 65536.0f) >= p) ? 1.f : 0.f;
        k[2 * i + 1] = ((float)(r[i] >> 16) * (1.0f / 65536.0f) >= p) ? 1.f : 0.f;
    }
}

// two per-channel sums of a CTA -> fp64 global accumulators.  Lanes that own the same channel chunk
// (lane % G) are folded by xor-shuffles first, so shared memory sees one atomic per warp per channel.  The CTAs
// of a cluster (8) are then folded through distributed shared memory by their rank-0 CTA, so a global address
// receives one fp64 atomic per CLUSTER: same-address atomics serialise in L2 (~30 cycles each), and with one per
// CTA the ~600 of them were a 5-8 us tail on every one of the ~290 statistics launches of an iteration.
// (Measured: the statistics kernel gains 11 %; the heavier backward-reduce kernel -- 122 registers -- LOSES 35 % when
// launched in clusters, so it keeps one atomic per CTA.)
constexpr int CLUSTER = 8;
template <bool CLUSTERED>
__device__ __forceinline__ void cta_accumulate(float (&a)[8], float (&b)[8], int G, float* s_a, float* s_b,
                                               double* g_a, double* g_b) {
    namespace cg = cooperative_groups;
    const int C = 8 * G;
    for (int c = threadIdx.x; c < C; c += BT) { s_a[c] = 0.f; s_b[c] = 0.f; }
    __syncthreads();
    for (int o = G; o < kWarp; o <<= 1) {
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            a[i] += __shfl_xor_sync(0xffffffffu, a[i], o);
            b[i] += __shfl_xor_sync(0xffffffffu, b[i], o);
        }
    }
    const int lane = threadIdx.x & 31;
    if (lane < G) {
#pragma unroll
        for (int i = 0; i < 8; ++i) { atomicAdd(s_a + lane * 8 + i, a[i]); atomicAdd(s_b + lane * 8 + i, b[i]); }
    }
    if constexpr (!CLUSTERED) {
        __syncthreads();
        for (int c = threadIdx.x; c < C; c += BT) { atomicAdd(g_a + c, (double)s_a[c]); atomicAdd(g_b + c, (double)s_b[c]); }
        return;
    }
    cg::cluster_group cluster = cg::this_cluster();
    cluster.sync();                                   // every CTA's shared-memory sums are complete and visible
    if (cluster.block_rank() == 0) {
        for (int c = threadIdx.x; c < C; c += BT) {
            double ra = 0.0, rb = 0.0;
            for (unsigned r = 0; r < cluster.num_blocks(); ++r) {
                ra += (double)*cluster.map_shared_rank(s_a + c, r);
                rb += (double)*cluster.map_shared_rank(s_b + c, r);
            }
            atomicAdd(g_a + c, ra);
            atomicAdd(g_b + c, rb);
        }
    }
    cluster.sync();                                   // peers keep their shared memory alive until rank 0 has read it
}

// Grid-stride loop with U independent 16-byte loads in flight per thread before any is consumed: at ~80 registers
// these kernels run 3 CTAs/SM, and one load per thread per iteration leaves HBM under-subscribed (measured 2.6-3.6 TB/s).
// `load(t)` returns the packet of element t, `use(t, packet)` consumes it.
template <int U, class Load, class Use>
__device__ __forceinline__ void stream_chunks(long long total, Load load, Use use) {
    const long long stride = (long long)gridDim.x * BT;
    long long t = (long long)blockIdx.x * BT + threadIdx.x;
    for (; t + (U - 1) * stride < total; t += U * stride) {
        decltype(load(t)) pk[U];
#pragma unroll
        for (int u = 0; u < U; ++u) pk[u] = load(t + u * stride);
#pragma unroll
        for (int u = 0; u < U; ++u) use(t + u * stride, pk[u]);
    }
    for (; t < total; t += stride) use(t, load(t));
}
struct Pair16 { uint4 g, y; };

__global__ void __cluster_dims__(CLUSTER, 1, 1) __launch_bounds__(BT) bn_stats_kernel(const uint4* __restrict__ y, long long npix, int G,
                                                      double* __restrict__ sum, double* __restrict__ sumsq) {
    __shared__ float s_a[256], s_b[256];
    grid_dep_launch();
    grid_dep_wait();
    const long long total = npix * G;
    float a[8], b[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) a[i] = b[i] = 0.f;
    stream_chunks<4>(total, [&](long long t) { return __ldg(y + t); }, [&](long long, const uint4& r) {
        float v[8];
        unpack8(r, v);
#pragma unroll
        for (int i = 0; i < 8; ++i) { a[i] += v[i]; b[i] = fmaf(v[i], v[i], b[i]); }
    });
    cta_accumulate<true>(a, b, G, s_a, s_b, sum, sumsq);
}

struct BnParams {
    const double* sum; const double* sumsq;       // forward: batch sums; backward: sum(g'), sum(g' * xhat)
    const float* gamma; const float* beta;
    float* running_mean; float* running_var;      // updated by CTA 0 in forward (nullable)
    float* save_mean; float* save_rstd;           // forward: written by CTA 0; backward: read
    float momentum, eps, slope, p, keep_scale;
    uint64_t seed;
    long long npix;
    int G;
    float* dgamma_accum; float* dbeta_accum;      // backward: optional fp32 gradient buffers to accumulate into
    const uint64_t* seed_dev;                     // nullable: per-iteration key added to `seed` (UapsStepState.key_rank)
    int nrep;                                     // forward: the batch sums arrive as nrep replicas of [sum[C] | sumsq[C]] to be added
};
__device__ __forceinline__ uint64_t eff_seed(const BnParams& p) { return p.seed + (p.seed_dev != nullptr ? *p.seed_dev : 0ull); }

// z = y * sc + sh with sc = gamma * rstd, sh = beta - mean * sc, from the SAVED fp32 mean / rstd and rounded the same way in
// the forward and both backward kernels: an element whose z lies within an ulp of 0 then takes one LeakyReLU branch in
// all three (three differently rounded shifts disagreed in about a third of the channels, so such an element could be
// differentiated on the other branch than the one the forward took).
__device__ __forceinline__ void bn_scale_shift(float gamma, float beta, float mean, float rstd, float& sc, float& sh) {
    sc = __fmul_rn(gamma, rstd);
    sh = __fmaf_rn(-mean, sc, beta);
}

// forward: a = dropout(leaky_relu(gamma * (y - mean) * rstd + beta))
__global__ void __launch_bounds__(BT) bn_act_kernel(const uint4* __restrict__ y, uint4* __restrict__ out, const BnParams p) {
    __shared__ float s_scale[256], s_shift[256];
    grid_dep_launch();
    grid_dep_wait();
    const int C = 8 * p.G;
    const double n = (double)p.npix;
    for (int c = threadIdx.x; c < C; c += BT) {
        double s1 = 0.0, s2 = 0.0;
        for (int r = 0; r < p.nrep; ++r) { s1 += p.sum[(size_t)r * 2 * C + c]; s2 += p.sumsq[(size_t)r * 2 * C + c]; }
        const double mean = s1 / n;
        double var = s2 / n - mean * mean;
        if (var < 0.0) var = 0.0;
        const float rstd = (float)(1.0 / sqrt(var + (double)p.eps));
        bn_scale_shift(p.gamma[c], p.beta[c], (float)mean, rstd, s_scale[c], s_shift[c]);
        if (blockIdx.x == 0) {
            p.save_mean[c] = (float)mean;
            p.save_rstd[c] = rstd;
            if (p.running_mean != nullptr) {
                const double unbiased = n > 1.0 ? var * n / (n - 1.0) : var;
                p.running_mean[c] = (1.f - p.momentum) * p.running_mean[c] + p.momentum * (float)mean;
                p.running_var[c] = (1.f - p.momentum) * p.running_var[c] + p.momentum * (float)unbiased;
            }
        }
    }
    __syncthreads();
    const int chunk = threadIdx.x % p.G;
    const uint64_t seed = p.p > 0.f ? eff_seed(p) : 0ull;
    float sc[8], sh[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) { sc[i] = s_scale[chunk * 8 + i]; sh[i] = s_shift[chunk * 8 + i]; }
    const long long total = p.npix * p.G;
    stream_chunks<4>(total, [&](long long t) { return __ldg(y + t); }, [&](long long t, const uint4& r) {
        float v[8], k[8];
        unpack8(r, v);
        if (p.p > 0.f) keep8(seed, (uint64_t)t, p.p, k);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            float z = fmaf(v[i], sc[i], sh[i]);
            z = z > 0.f ? z : z * p.slope;
            if (p.p > 0.f) z *= k[i] * p.keep_scale;
            v[i] = z;
        }
        out[t] = pack8(v);
    });
}

// g' = g * dropout' * leaky_relu'(z); accumulate sum(g') and sum(g' * y) per channel.
// The kernels are instruction-issue bound (ncu: 64 % issue-active at 23 % occupancy, profiles/r02_kernels_a.txt), so the
// per-element work is folded into per-channel constants: z = y * sc + sh with sc = gamma * rstd, sh = beta - mean * sc
// (one FMA instead of subtract / multiply / FMA), and the RAW second moment sum(g' * y) is accumulated -- the consumer
// recovers sum(g' * xhat) = rstd * (sum(g' * y) - mean * sum(g')) in fp64.
template <int U, int MINB>
__global__ void __launch_bounds__(BT, MINB) bn_act_bwd_reduce_kernel(const uint4* __restrict__ g, const uint4* __restrict__ y,
                                                                  const BnParams p, double* __restrict__ sum_g,
                                                                  double* __restrict__ sum_gy) {
    __shared__ float s_a[256], s_b[256];
    grid_dep_launch();
    grid_dep_wait();
    const int chunk = threadIdx.x % p.G;
    const uint64_t seed = p.p > 0.f ? eff_seed(p) : 0ull;
    float sc[8], sh[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const int c = chunk * 8 + i;
        bn_scale_shift(p.gamma[c], p.beta[c], p.save_mean[c], p.save_rstd[c], sc[i], sh[i]);
    }
    // packed fp32x2 arithmetic (FFMA2 / FMUL2 / FADD2, IEEE per lane: the same values as the scalar form): a bf16x2 pair
    // converts straight into a float2 and the five arithmetic instructions per element become five per pair
    float2 sc2[4], sh2[4], a2[4], b2[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        sc2[i] = make_float2(sc[2 * i], sc[2 * i + 1]);
        sh2[i] = make_float2(sh[2 * i], sh[2 * i + 1]);
        a2[i] = b2[i] = make_float2(0.f, 0.f);
    }
    const float2 slope2 = make_float2(p.slope, p.slope);
    const bool drop = p.p > 0.f;
    const long long total = p.npix * p.G;
    stream_chunks<U>(total, [&](long long t) { return Pair16{__ldg(g + t), __ldg(y + t)}; }, [&](long long t, const Pair16& pk) {
        float k[8];
        if (drop) keep8(seed, (uint64_t)t, p.p, k);
        const __nv_bfloat162* gh = reinterpret_cast<const __nv_bfloat162*>(&pk.g);
        const __nv_bfloat162* yh = reinterpret_cast<const __nv_bfloat162*>(&pk.y);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const float2 gv = __bfloat1622float2(gh[i]), v = __bfloat1622float2(yh[i]);
            const float2 z = __ffma2_rn(v, sc2[i], sh2[i]);
            const float2 gs = __fmul2_rn(gv, slope2);
            float2 gp = make_float2(z.x > 0.f ? gv.x : gs.x, z.y > 0.f ? gv.y : gs.y);
            if (drop) gp = __fmul2_rn(gp, make_float2(k[2 * i] * p.keep_scale, k[2 * i + 1] * p.keep_scale));
            a2[i] = __fadd2_rn(a2[i], gp);
            b2[i] = __ffma2_rn(gp, v, b2[i]);
        }
    });
    float a[8], b[8];
#pragma unroll
    for (int i = 0; i < 4; ++i) { a[2 * i] = a2[i].x; a[2 * i + 1] = a2[i].y; b[2 * i] = b2[i].x; b[2 * i + 1] = b2[i].y; }
    cta_accumulate<false>(a, b, p.G, s_a, s_b, sum_g, sum_gy);
}

// dy = gamma * rstd * (g' - mean(g') - xhat * mean(g' * xhat)) = g' * A + y * Bc + Cc with per-channel
//   A = gamma * rstd, Bc = -A * rstd * mgx, Cc = A * (mean * rstd * mgx - mg),  mg = sum(g') / n,  mgx = sum(g' * xhat) / n
template <int U, int MINB>
__global__ void __launch_bounds__(BT, MINB) bn_act_bwd_kernel(const uint4* __restrict__ g, const uint4* __restrict__ y,
                                                           uint4* __restrict__ dy, const BnParams p) {
    __shared__ float s_A[256], s_sh[256], s_B[256], s_C[256];
    grid_dep_launch();
    grid_dep_wait();
    const int C = 8 * p.G;
    const double invn = 1.0 / (double)p.npix;
    for (int c = threadIdx.x; c < C; c += BT) {
        const double mean = (double)p.save_mean[c], rstd = (double)p.save_rstd[c], ga = (double)p.gamma[c];
        const double sg = p.sum[c], sgx = rstd * (p.sumsq[c] - mean * sg);      // sum(g'), sum(g' * xhat)
        const double A = ga * rstd, mg = sg * invn, mgx = sgx * invn;
        bn_scale_shift(p.gamma[c], p.beta[c], p.save_mean[c], p.save_rstd[c], s_A[c], s_sh[c]);   // (float)A == s_A[c]
        s_B[c] = (float)(-A * rstd * mgx);
        s_C[c] = (float)(A * (mean * rstd * mgx - mg));
        if (blockIdx.x == 0 && p.dgamma_accum != nullptr) {   // d gamma = sum(g' * xhat), d beta = sum(g'): add to .grad
            p.dgamma_accum[c] += (float)sgx;
            p.dbeta_accum[c] += (float)sg;
        }
    }
    __syncthreads();
    const int chunk = threadIdx.x % p.G;
    const uint64_t seed = p.p > 0.f ? eff_seed(p) : 0ull;
    float A[8], sh[8], Bc[8], Cc[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const int c = chunk * 8 + i;
        A[i] = s_A[c]; sh[i] = s_sh[c]; Bc[i] = s_B[c]; Cc[i] = s_C[c];
    }
    const long long total = p.npix * p.G;
    stream_chunks<U>(total, [&](long long t) { return Pair16{__ldg(g + t), __ldg(y + t)}; }, [&](long long t, const Pair16& pk) {
        float gv[8], v[8], k[8];
        unpack8(pk.g, gv);
        unpack8(pk.y, v);
        if (p.p > 0.f) keep8(seed, (uint64_t)t, p.p, k);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const float z = fmaf(v[i], A[i], sh[i]);
            float gp = gv[i] * (z > 0.f ? 1.f : p.slope);
            if (p.p > 0.f) gp *= k[i] * p.keep_scale;
            v[i] = fmaf(gp, A[i], fmaf(v[i], Bc[i], Cc[i]));
        }
        dy[t] = pack8(v);
    });
}

inline int bn_grid(long long chunks, int ctas_per_sm = 8) {
    static const int mult = [] { const char* e = getenv("UAPS_BN_GRID_MULT"); return e ? atoi(e) : 1; }();   // A/B knob: waves per launch
    long long want = ceil_div<long long>(chunks, BT), cap = (long long)device_info().sm_count * ctas_per_sm * (mult > 0 ? mult : 1);
    return (int)(want < cap ? (want < 1 ? 1 : want) : cap);
}
// the reducing kernels are launched in clusters: whole clusters only (surplus CTAs contribute zeros)
inline int bn_grid_clustered(long long chunks, int ctas_per_sm) {
    const int g = bn_grid(chunks, ctas_per_sm);
    return (g + CLUSTER - 1) / CLUSTER * CLUSTER;
}
inline bool valid_c(int C) { const int G = C / 8; return C % 8 == 0 && G >= 1 && G <= 32 && (G & (G - 1)) == 0; }

}  // namespace
}  // namespace uaps

using namespace uaps;

UAPS_API int uaps_bn_stats_nhwc(const void* y, int64_t npix, int C, double* sum, double* sumsq, cudaStream_t stream) {
    if (y == nullptr || sum == nullptr || sumsq == nullptr || npix <= 0) return UAPS_EINVAL;
    if (!valid_c(C)) return UAPS_ERANGE;
    if (!aligned_to(y, 16) || !aligned_to(sum, 8) || !aligned_to(sumsq, 8)) return UAPS_EALIGN;
    UAPS_LAUNCH(bn_stats_kernel, dim3(bn_grid_clustered(npix * (C / 8), 4)), dim3(BT), 0, stream, reinterpret_cast<const uint4*>(y),
                (long long)npix, C / 8, sum, sumsq);
    UAPS_LAUNCH_CHECK();
    return UAPS_OK;
}

UAPS_API int uaps_bn_act_nhwc(const void* y, const double* sum, const double* sumsq, const float* gamma, const float* beta,
                              float* running_mean, float* running_var, float momentum, float eps, float slope, double p_drop,
                              uint64_t seed, void* out, float* save_mean, float* save_rstd, int64_t npix, int C,
                              const uint64_t* seed_dev, int nrep, cudaStream_t stream) {
    if (y == nullptr || sum == nullptr || sumsq == nullptr || gamma == nullptr || beta == nullptr || out == nullptr ||
        save_mean == nullptr || save_rstd == nullptr || npix <= 0)
        return UAPS_EINVAL;
    if (!valid_c(C) || !(p_drop >= 0.0 && p_drop < 1.0) || nrep < 1 || nrep > 64) return UAPS_ERANGE;
    if (!aligned_to(y, 16) || !aligned_to(out, 16)) return UAPS_EALIGN;
    BnParams p{};
    p.nrep = nrep;                                // replica r: sum at sum[r * 2C + c], sumsq at sumsq[r * 2C + c]
    p.sum = sum; p.sumsq = sumsq; p.gamma = gamma; p.beta = beta; p.running_mean = running_mean; p.running_var = running_var;
    p.save_mean = save_mean; p.save_rstd = save_rstd; p.momentum = momentum; p.eps = eps; p.slope = slope; p.p = (float)p_drop;
    p.keep_scale = (float)(1.0 / (double)(float)(1.0 - p_drop)); p.seed = seed; p.npix = npix; p.G = C / 8;
    p.seed_dev = seed_dev;
    UAPS_LAUNCH(bn_act_kernel, dim3(bn_grid(npix * (C / 8), 4)), dim3(BT), 0, stream, reinterpret_cast<const uint4*>(y),
                reinterpret_cast<uint4*>(out), p);
    UAPS_LAUNCH_CHECK();
    return UAPS_OK;
}

UAPS_API int uaps_bn_act_bwd_nhwc(const void* g_out, const void* y, const float* gamma, const float* beta, const float* save_mean,
                                  const float* save_rstd, float slope, double p_drop, uint64_t seed, double* sum_g,
                                  double* sum_gx, void* dy, float* dgamma_accum, float* dbeta_accum, int64_t npix, int C,
                                  const uint64_t* seed_dev, cudaStream_t stream) {
    if (g_out == nullptr || y == nullptr || gamma == nullptr || beta == nullptr || save_mean == nullptr || save_rstd == nullptr ||
        sum_g == nullptr || sum_gx == nullptr || dy == nullptr || npix <= 0)
        return UAPS_EINVAL;
    if (!valid_c(C) || !(p_drop >= 0.0 && p_drop < 1.0)) return UAPS_ERANGE;
    if (!aligned_to(g_out, 16) || !aligned_to(y, 16) || !aligned_to(dy, 16)) return UAPS_EALIGN;
    BnParams p{};
    p.sum = sum_g; p.sumsq = sum_gx; p.gamma = gamma; p.beta = beta; p.save_mean = const_cast<float*>(save_mean);
    p.save_rstd = const_cast<float*>(save_rstd); p.slope = slope; p.p = (float)p_drop;
    p.keep_scale = (float)(1.0 / (double)(float)(1.0 - p_drop)); p.seed = seed; p.npix = npix; p.G = C / 8;
    if ((dgamma_accum == nullptr) != (dbeta_accum == nullptr)) return UAPS_EINVAL;
    p.dgamma_accum = dgamma_accum; p.dbeta_accum = dbeta_accum; p.seed_dev = seed_dev;
    // sum_g / sum_gx (zeroed by the caller) receive sum(g') and the RAW sum(g' * y); the second kernel turns the latter into
    // sum(g' * xhat) = d gamma.  Variant = (loads in flight per thread, resident CTAs / SM); UAPS_BN_BWD_VARIANT picks (A/B knob).
    static const int variant = [] { const char* e = getenv("UAPS_BN_BWD_VARIANT"); return e ? atoi(e) : 1; }();
    const uint4* g4 = reinterpret_cast<const uint4*>(g_out);
    const uint4* y4 = reinterpret_cast<const uint4*>(y);
    uint4* dy4 = reinterpret_cast<uint4*>(dy);
    const long long chunks = npix * (C / 8);
#define UAPS_BN_BWD(U1, M1, U2, M2)                                                                          \
    UAPS_LAUNCH((bn_act_bwd_reduce_kernel<U1, M1>), dim3(bn_grid(chunks, M1)), dim3(BT), 0, stream, g4, y4, p, sum_g, sum_gx); \
    UAPS_LAUNCH_CHECK();                                                                                     \
    UAPS_LAUNCH((bn_act_bwd_kernel<U2, M2>), dim3(bn_grid(chunks, M2)), dim3(BT), 0, stream, g4, y4, dy4, p);
    if (variant == 0) { UAPS_BN_BWD(4, 2, 2, 2) }
    else if (variant == 1) { UAPS_BN_BWD(3, 3, 2, 3) }
    else if (variant == 3) { UAPS_BN_BWD(2, 4, 2, 4) }
    else { UAPS_BN_BWD(2, 3, 2, 3) }
#undef UAPS_BN_BWD
    UAPS_LAUNCH_CHECK();
    return UAPS_OK;
}
