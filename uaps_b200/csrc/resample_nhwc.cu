// Bilinear x2 upsampling with align_corners=True (nn.Upsample in UpBlock, utilities/UAPS_unet.py:74-75,84)
// and 2x2 max pooling (nn.MaxPool2d(2) in DownBlock, :56) on channels-last bf16 activations, forward and
// backward.  One thread owns a 16-byte chunk (8 channels) of one OUTPUT pixel (forward) or one INPUT
// pixel (backward: gather form, no atomics), so every access is a full 16-byte vector and a warp
// covers 512 contiguous bytes.
#include <cuda_bf16.h>
#include "common.cuh"

namespace uaps {
namespace {

constexpr int RT = 256;

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

// source coordinate of output index o: o * (in-1)/(out-1)  (align_corners=True), as torch computes it in fp32
__device__ __forceinline__ void src_coord(int o, float scale, int in_size, int& i0, int& i1, float& l1) {
    const float s = scale * o;
    i0 = (int)s;
    if (i0 > in_size - 1) i0 = in_size - 1;
    i1 = i0 + (i0 < in_size - 1 ? 1 : 0);
    l1 = s - (float)i0;
}

// Both resampling kernels use a 3-D grid -- x: 16-byte chunks along a row (pixel * G + g), y: INPUT rows in bands of
// RY, z: image -- so the index math is 32-bit and a CTA covers a 2-D patch whose stencils overlap in L1.
// Round 2: ncu showed both kernels instruction-issue bound (75-77 % issue-active at 1.8-2.3 TB/s,
// profiles/r02_kernels_ncu_full.txt), so the per-output instruction count was cut:
//   * packed fp32x2 arithmetic (FFMA2 / FMUL2, sm_100): a bf16x2 pair converts straight into a float2 and the
//     interpolation runs on pairs -- half the FMA-pipe instructions, IEEE per lane (results unchanged);
//   * forward: a thread produces the TWO output rows 2k, 2k+1 of its column; their source rows are always drawn from
//     {y0(2k), y1(2k), y1(2k+1)} (checked exhaustively in fp32 for every size up to 1024), so three horizontally
//     interpolated rows serve both outputs: 6 loads and 40 packed operations per 2 outputs instead of 8 and 96 scalar;
//   * backward: the outputs that tap input i are exactly o in [2i-1, 2i+2] (checked the same way): 4 x 4 candidates instead
//     of 6 x 6 with per-candidate branches, and their weights come from a small shared-memory table computed once per CTA.
constexpr int RX = 32, RY = 8;            // CTA = 32 chunks x 8 rows = 256 threads

__device__ __forceinline__ void unpack4(const uint4& r, float2 (&v)[4]) {
    const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&r);
#pragma unroll
    for (int i = 0; i < 4; ++i) v[i] = __bfloat1622float2(h[i]);
}
__device__ __forceinline__ uint4 pack4(const float2 (&v)[4]) {
    uint4 r;
    __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(&r);
#pragma unroll
    for (int i = 0; i < 4; ++i) h[i] = __float22bfloat162_rn(v[i]);
    return r;
}
// horizontally interpolated row: hx * left + lx * right (the rounding order of the scalar expression it replaces)
__device__ __forceinline__ void hrow(const uint4* __restrict__ row, unsigned off0, unsigned off1, float2 hx, float2 lx, float2 (&h)[4]) {
    float2 a[4], c[4];
    unpack4(__ldg(row + off0), a);
    unpack4(__ldg(row + off1), c);
#pragma unroll
    for (int i = 0; i < 4; ++i) h[i] = __ffma2_rn(c[i], lx, __fmul2_rn(a[i], hx));
}

__global__ void __launch_bounds__(RT) upsample2x_fwd_kernel(const uint4* __restrict__ x, uint4* __restrict__ y, int H, int W,
                                                            int G, float sh, float sw) {
    grid_dep_launch();
    grid_dep_wait();
    const int OW = 2 * W;
    const unsigned col = blockIdx.x * RX + threadIdx.x;           // output chunk column: ox * G + g
    const int k = blockIdx.y * RY + threadIdx.y;                  // input row band: output rows 2k and 2k + 1
    if (col >= (unsigned)OW * G || k >= H) return;
    const int ox = col / G, g = col - ox * G;
    int x0, x1, y0a, y1a, y0b, y1b; float lxs, lya, lyb;
    src_coord(ox, sw, W, x0, x1, lxs);
    src_coord(2 * k, sh, H, y0a, y1a, lya);                       // warp-uniform (a warp spans x only)
    src_coord(2 * k + 1, sh, H, y0b, y1b, lyb);
    const uint4* xb = x + (size_t)blockIdx.z * H * W * G + g;
    const unsigned o0 = (unsigned)x0 * G, o1 = (unsigned)x1 * G, rowp = (unsigned)W * G;
    const float2 lx = make_float2(lxs, lxs), hx = make_float2(1.f - lxs, 1.f - lxs);
    float2 h0[4], h1[4], h2[4], o[4];
    hrow(xb + (size_t)y0a * rowp, o0, o1, hx, lx, h0);
    hrow(xb + (size_t)y1a * rowp, o0, o1, hx, lx, h1);
    {
        const float2 ly = make_float2(lya, lya), hy = make_float2(1.f - lya, 1.f - lya);
#pragma unroll
        for (int i = 0; i < 4; ++i) o[i] = __ffma2_rn(h1[i], ly, __fmul2_rn(h0[i], hy));
        y[((size_t)blockIdx.z * 2 * H + 2 * k) * OW * G + col] = pack4(o);
    }
    // second output row: its upper tap is y0a or y1a (always), its lower tap y1a or a new row
    if (y1b != y1a) hrow(xb + (size_t)y1b * rowp, o0, o1, hx, lx, h2);
    {
        const float2 ly = make_float2(lyb, lyb), hy = make_float2(1.f - lyb, 1.f - lyb);
        const bool up_is_a0 = (y0b == y0a), lo_is_a1 = (y1b == y1a);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const float2 up = up_is_a0 ? h0[i] : h1[i];
            const float2 lo = lo_is_a1 ? h1[i] : h2[i];
            o[i] = __ffma2_rn(lo, ly, __fmul2_rn(up, hy));
        }
        y[((size_t)blockIdx.z * 2 * H + 2 * k + 1) * OW * G + col] = pack4(o);
    }
}

// weight of output index o onto input index i along one axis (0 when o's two taps miss i or o is out of range)
__device__ __forceinline__ float tap_weight(int o, int i, float scale, int in_size) {
    if (o < 0 || o >= 2 * in_size) return 0.f;
    int i0, i1; float l1;
    src_coord(o, scale, in_size, i0, i1, l1);
    return (i0 == i ? 1.f - l1 : 0.f) + (i1 == i ? l1 : 0.f);
}

// gather backward: input pixel (iy, ix) collects from the outputs whose stencil touches it: o in [2i-1, 2i+2] per axis
// (the fp32 evaluation of o * r is the forward's, so borderline taps land where the forward put them).
constexpr int NCAND = 4;
__global__ void __launch_bounds__(RT) upsample2x_bwd_kernel(const uint4* __restrict__ gy, uint4* __restrict__ gx, int H, int W,
                                                            int G, float sh, float sw) {
    __shared__ float s_wy[RY][NCAND];
    __shared__ float s_wx[RX][NCAND];                             // one entry per pixel column of the CTA (<= RX when G = 1)
    grid_dep_launch();
    grid_dep_wait();
    const int OH = 2 * H, OW = 2 * W;
    const int t = threadIdx.y * RX + threadIdx.x;
    const int px0 = (blockIdx.x * RX) / G;                        // first pixel column of this CTA
    if (t < RY * NCAND) {
        const int r = t / NCAND, a = t % NCAND, iy = blockIdx.y * RY + r;
        s_wy[r][a] = iy < H ? tap_weight(2 * iy - 1 + a, iy, sh, H) : 0.f;
    } else if (t >= 64 && t < 64 + RX * NCAND) {
        const int q = (t - 64) / NCAND, b = (t - 64) % NCAND, ix = px0 + q;
        s_wx[q][b] = ix < W ? tap_weight(2 * ix - 1 + b, ix, sw, W) : 0.f;
    }
    __syncthreads();
    const unsigned col = blockIdx.x * RX + threadIdx.x;
    const int iy = blockIdx.y * RY + threadIdx.y;
    if (col >= (unsigned)W * G || iy >= H) return;
    const int ix = col / G, g = col - ix * G;
    float wy[NCAND], wx[NCAND];
#pragma unroll
    for (int a = 0; a < NCAND; ++a) { wy[a] = s_wy[threadIdx.y][a]; wx[a] = s_wx[ix - px0][a]; }
    float2 acc[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) acc[i] = make_float2(0.f, 0.f);
    const uint4* gb = gy + (size_t)blockIdx.z * OH * OW * G + g;
#pragma unroll
    for (int a = 0; a < NCAND; ++a) {
        int oy = 2 * iy - 1 + a;
        oy = oy < 0 ? 0 : (oy >= OH ? OH - 1 : oy);               // out-of-range candidates have zero weight: clamp the address
        const uint4* row = gb + (size_t)oy * OW * G;
#pragma unroll
        for (int b = 0; b < NCAND; ++b) {
            int ox = 2 * ix - 1 + b;
            ox = ox < 0 ? 0 : (ox >= OW ? OW - 1 : ox);
            float2 v[4];
            unpack4(__ldg(row + (unsigned)ox * G), v);
            const float w = wy[a] * wx[b];
            const float2 w2 = make_float2(w, w);
#pragma unroll
            for (int i = 0; i < 4; ++i) acc[i] = __ffma2_rn(v[i], w2, acc[i]);
        }
    }
    gx[((size_t)blockIdx.z * H + iy) * W * G + col] = pack4(acc);
}

// [B,C,H,W] fp32 (NCHW) -> [B,H,W,Cp] bf16 (channels-last, channels C..Cp-1 zero): the network input and the
// logits gradient entering the bf16 path.  One thread per pixel: per channel a warp reads 128 contiguous bytes.
__global__ void __launch_bounds__(RT) nchw_f32_to_nhwc_bf16_kernel(const float* __restrict__ x, uint4* __restrict__ out, int C,
                                                                   int HW, int Gp) {
    grid_dep_launch();
    grid_dep_wait();
    const int p = blockIdx.x * RT + threadIdx.x;
    if (p >= HW) return;
    const float* xb = x + (size_t)blockIdx.y * C * HW + p;
    uint4* ob = out + ((size_t)blockIdx.y * HW + p) * Gp;
    for (int g = 0; g < Gp; ++g) {
        float v[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int c = g * 8 + i;
            v[i] = c < C ? __ldg(xb + (size_t)c * HW) : 0.f;
        }
        ob[g] = pack8(v);
    }
}

// The same conversion for the logits gradient, which also accumulates the per-channel sums of the (bf16-rounded) values it
// writes -- the bias gradient of out_conv (UAPS_unet.py:138-139) -- so that the separate reduction pass over the padded
// 16-channel tensor is not needed.  C <= 8; sums: NREP replicas of [Cp] doubles, zeroed by the caller (replica
// blockIdx.x % NREP: same-address fp64 atomics serialise in L2).
constexpr int ENTRY_NREP = 16;
__global__ void __launch_bounds__(RT) nchw_f32_to_nhwc_bf16_sums_kernel(const float* __restrict__ x, uint4* __restrict__ out, int C,
                                                                        int HW, int Gp, double* __restrict__ sums) {
    __shared__ float s_part[RT / 32][8];
    grid_dep_launch();
    grid_dep_wait();
    const int p = blockIdx.x * RT + threadIdx.x;
    float v[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] = 0.f;
    if (p < HW) {
        const float* xb = x + (size_t)blockIdx.y * C * HW + p;
        uint4* ob = out + ((size_t)blockIdx.y * HW + p) * Gp;
#pragma unroll
        for (int i = 0; i < 8; ++i)
            if (i < C) v[i] = __bfloat162float(__float2bfloat16_rn(__ldg(xb + (size_t)i * HW)));   // what the tensor will hold
        ob[0] = pack8(v);
        for (int g = 1; g < Gp; ++g) ob[g] = make_uint4(0u, 0u, 0u, 0u);
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v[i] += __shfl_xor_sync(0xffffffffu, v[i], o);
    }
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (lane == 0) {
#pragma unroll
        for (int i = 0; i < 8; ++i) s_part[warp][i] = v[i];
    }
    __syncthreads();
    if (threadIdx.x < C) {
        float t = 0.f;
#pragma unroll
        for (int w = 0; w < RT / 32; ++w) t += s_part[w][threadIdx.x];
        atomicAdd(sums + (size_t)(blockIdx.x % ENTRY_NREP) * (Gp * 8) + threadIdx.x, (double)t);
    }
}

// torch's max-pool rule (nn.MaxPool2d on CUDA): scanning the window in (row, column) order, a candidate replaces the running
// maximum when it is greater OR NaN -- so a NaN anywhere in the window propagates to the output (fmaxf would drop it, and a NaN
// activation would vanish at the pooling layer instead of reaching the loss)
__device__ __forceinline__ float pool_pick(float m, float v) { return (v > m || isnan(v)) ? v : m; }

__global__ void __launch_bounds__(RT) maxpool2_fwd_kernel(const uint4* __restrict__ x, uint4* __restrict__ y, int B, int H, int W, int G) {
    grid_dep_launch();
    grid_dep_wait();
    const int OH = H / 2, OW = W / 2;
    const long long total = (long long)B * OH * OW * G;
    for (long long t = (long long)blockIdx.x * RT + threadIdx.x; t < total; t += (long long)gridDim.x * RT) {
        const int g = (int)(t % G);
        long long p = t / G;
        const int ox = (int)(p % OW); p /= OW;
        const int oy = (int)(p % OH);
        const int b = (int)(p / OH);
        const uint4* xb = x + ((size_t)b * H * W + (size_t)(2 * oy) * W + 2 * ox) * G + g;
        float a[8], c[8], d[8], e[8];
        unpack8(__ldg(xb), a); unpack8(__ldg(xb + G), c);
        unpack8(__ldg(xb + (size_t)W * G), d); unpack8(__ldg(xb + (size_t)W * G + G), e);
#pragma unroll
        for (int i = 0; i < 8; ++i) a[i] = pool_pick(pool_pick(pool_pick(a[i], c[i]), d[i]), e[i]);
        y[t] = pack8(a);
    }
}

// the gradient goes to the element the forward picked (pool_pick in (row, column) order: the first maximum, or the last NaN),
// as torch's max_pool2d backward does
__global__ void __launch_bounds__(RT) maxpool2_bwd_kernel(const uint4* __restrict__ x, const uint4* __restrict__ gy,
                                                          uint4* __restrict__ gx, int B, int H, int W, int G) {
    grid_dep_launch();
    grid_dep_wait();
    const int OH = H / 2, OW = W / 2;
    const long long total = (long long)B * OH * OW * G;
    for (long long t = (long long)blockIdx.x * RT + threadIdx.x; t < total; t += (long long)gridDim.x * RT) {
        const int g = (int)(t % G);
        long long p = t / G;
        const int ox = (int)(p % OW); p /= OW;
        const int oy = (int)(p % OH);
        const int b = (int)(p / OH);
        const size_t base = ((size_t)b * H * W + (size_t)(2 * oy) * W + 2 * ox) * G + g;
        const size_t offs[4] = {0, (size_t)G, (size_t)W * G, (size_t)W * G + G};
        float v[4][8], gv[8], o[4][8];
#pragma unroll
        for (int k = 0; k < 4; ++k) unpack8(__ldg(x + base + offs[k]), v[k]);
        unpack8(__ldg(gy + t), gv);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            int best = 0;
            float m = v[0][i];
#pragma unroll
            for (int k = 1; k < 4; ++k)
                if (v[k][i] > m || isnan(v[k][i])) { m = v[k][i]; best = k; }
#pragma unroll
            for (int k = 0; k < 4; ++k) o[k][i] = (k == best) ? gv[i] : 0.f;
        }
#pragma unroll
        for (int k = 0; k < 4; ++k) gx[base + offs[k]] = pack8(o[k]);
    }
}

inline int rgrid(long long n) {
    long long want = ceil_div<long long>(n, RT), cap = (long long)device_info().sm_count * 8;
    return (int)(want < cap ? (want < 1 ? 1 : want) : cap);
}

}  // namespace
}  // namespace uaps

using namespace uaps;

UAPS_API int uaps_upsample2x_nhwc(const void* x, void* y, int B, int H, int W, int C, int backward, cudaStream_t stream) {
    if (x == nullptr || y == nullptr || B <= 0 || H <= 0 || W <= 0) return UAPS_EINVAL;
    if (C % 8 != 0 || C <= 0) return UAPS_ERANGE;
    if (!aligned_to(x, 16) || !aligned_to(y, 16)) return UAPS_EALIGN;
    const int G = C / 8;
    const float sh = H > 1 ? (float)(H - 1) / (float)(2 * H - 1) : 0.f, sw = W > 1 ? (float)(W - 1) / (float)(2 * W - 1) : 0.f;
    if (B > 65535 || ceil_div(2 * H, RY) > 65535) return UAPS_ERANGE;
    const dim3 block(RX, RY);
    if (!backward)      // x: [B,H,W,C] -> y: [B,2H,2W,C]
        UAPS_LAUNCH(upsample2x_fwd_kernel, dim3(ceil_div(2 * W * G, RX), ceil_div(H, RY), B), block, 0, stream,
                    reinterpret_cast<const uint4*>(x), reinterpret_cast<uint4*>(y), H, W, G, sh, sw);
    else                // x: upstream gradient [B,2H,2W,C] -> y: [B,H,W,C]
        UAPS_LAUNCH(upsample2x_bwd_kernel, dim3(ceil_div(W * G, RX), ceil_div(H, RY), B), block, 0, stream,
                    reinterpret_cast<const uint4*>(x), reinterpret_cast<uint4*>(y), H, W, G, sh, sw);
    UAPS_LAUNCH_CHECK();
    return UAPS_OK;
}

UAPS_API int uaps_maxpool2_nhwc(const void* x, const void* gy, void* out, int B, int H, int W, int C, cudaStream_t stream) {
    if (x == nullptr || out == nullptr || B <= 0 || H <= 0 || W <= 0) return UAPS_EINVAL;
    if (C % 8 != 0 || C <= 0 || (H % 2) != 0 || (W % 2) != 0) return UAPS_ERANGE;
    if (!aligned_to(x, 16) || !aligned_to(out, 16) || !aligned_to(gy, 16)) return UAPS_EALIGN;
    const int G = C / 8;
    const long long n = (long long)B * (H / 2) * (W / 2) * G;
    if (gy == nullptr)  // forward: x [B,H,W,C] -> out [B,H/2,W/2,C]
        UAPS_LAUNCH(maxpool2_fwd_kernel, dim3(rgrid(n)), dim3(RT), 0, stream, reinterpret_cast<const uint4*>(x), reinterpret_cast<uint4*>(out), B, H, W, G);
    else                // backward: out = d x [B,H,W,C] (every element written)
        UAPS_LAUNCH(maxpool2_bwd_kernel, dim3(rgrid(n)), dim3(RT), 0, stream, reinterpret_cast<const uint4*>(x),
                    reinterpret_cast<const uint4*>(gy), reinterpret_cast<uint4*>(out), B, H, W, G);
    UAPS_LAUNCH_CHECK();
    return UAPS_OK;
}

UAPS_API int uaps_nchw_f32_to_nhwc_bf16(const float* x, void* out, int B, int C, int H, int W, int Cp, cudaStream_t stream) {
    if (x == nullptr || out == nullptr || B <= 0 || C <= 0 || H <= 0 || W <= 0) return UAPS_EINVAL;
    if (Cp % 8 != 0 || Cp < C || B > 65535 || (long long)H * W >= 2147483647LL) return UAPS_ERANGE;
    if (!aligned_to(x, 4) || !aligned_to(out, 16)) return UAPS_EALIGN;
    const int HW = H * W;
    UAPS_LAUNCH(nchw_f32_to_nhwc_bf16_kernel, dim3(ceil_div(HW, RT), B), dim3(RT), 0, stream, x, reinterpret_cast<uint4*>(out), C, HW, Cp / 8);
    UAPS_LAUNCH_CHECK();
    return UAPS_OK;
}

UAPS_API int uaps_nchw_f32_to_nhwc_bf16_sums_nrep(void) { return ENTRY_NREP; }

UAPS_API int uaps_nchw_f32_to_nhwc_bf16_sums(const float* x, void* out, int B, int C, int H, int W, int Cp, double* sums,
                                             cudaStream_t stream) {
    if (x == nullptr || out == nullptr || sums == nullptr || B <= 0 || C <= 0 || H <= 0 || W <= 0) return UAPS_EINVAL;
    if (C > 8 || Cp % 8 != 0 || Cp < C || B > 65535 || (long long)H * W >= 2147483647LL) return UAPS_ERANGE;
    if (!aligned_to(x, 4) || !aligned_to(out, 16) || !aligned_to(sums, 8)) return UAPS_EALIGN;
    const int HW = H * W;
    UAPS_LAUNCH(nchw_f32_to_nhwc_bf16_sums_kernel, dim3(ceil_div(HW, RT), B), dim3(RT), 0, stream, x, reinterpret_cast<uint4*>(out), C,
                HW, Cp / 8, sums);
    UAPS_LAUNCH_CHECK();
    return UAPS_OK;
}
