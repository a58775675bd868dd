// Implicit-GEMM convolution (3x3 pad 1 / 1x1, stride 1) on the 5th-gen tensor cores:
// tcgen05.mma with the accumulator in TMEM, activations fed by TMA, weights by bulk-async copies.
// Replaces the cuDNN calls behind nn.Conv2d in ConvBlock / UpBlock / out_conv of
// utilities/UAPS_unet.py:31-47, 65-86, 138-139 (forward), and -- with rotated/transposed packed
// weights -- their data-gradient.
//
// GEMM view: M = 128 output pixels (a 16 x 8 spatial tile of one image), N = output channels of
// this CTA (N_TILE <= 128), K = taps x input channels.  Activations are NHWC bf16.
//
//   A operand.  One TMA box {CK channels, 8 x, 16+2 y, 1 n} per horizontal tap s in {-1,0,+1} lands
//   as a K-major [144 rows][CK] tile whose rows are (y, x) and whose row pitch (CK*2 B) equals the
//   swizzle span.  Eight consecutive rows = one image row = exactly one swizzle atom, so the three
//   vertical taps r are the SAME tile read at row offsets 0 / 8 / 16: atom-aligned descriptor starts,
//   no re-load.  Out-of-image coordinates (incl. negative) are zero-filled by TMA = the conv padding.
//   3 loads serve 9 taps (3.4x operand traffic out of L2 instead of 9x).
//   A concatenated input (UpBlock's torch.cat([skip, up]), :85) is two K segments with two tensor
//   maps: the concat is never materialised.
//
//   B operand.  Weights are packed once per step into the exact shared-memory image
//   [n_tile][segment][chunk][s][r][N_TILE][CK] bf16 with the 16-byte swizzle already applied, so a
//   stage's three r-blocks are one contiguous cp.async.bulk.
//
//   D.  128 lanes x N_TILE fp32 columns of TMEM.  Epilogue: tcgen05.ld 32x32b, + bias, -> bf16 NHWC
//   (or fp32 NCHW for the logits that feed the fused loss kernel).
//
// Kernels.  conv_igemm_persistent_kernel (default): one CTA per SM slot (up to 6 per SM for the small layers) walks the
// output tiles with stride gridDim.x; 6 warps: warp 0 lane 0 = TMA producer running ahead through a 2-4 stage mbarrier
// ring, warp 1 lane 0 = MMA issuer alternating between two TMEM accumulators, warps 2-5 = epilogue (tcgen05.ld -> + bias
// [-> LeakyReLU] -> bf16 NHWC / fp32 NCHW), so tile i's epilogue overlaps tile i+1's MMAs.  Layers whose packed weights fit
// 80 KB keep them resident in shared memory and load ONE x-halo activation box per channel chunk for all nine taps.
// conv_sn_kernel (3x3 layers with <= 64 output channels and input channels >= 2x output channels or >= 64): the horizontal taps
// in the MMA's N dimension -- every A tile is fetched 3 times instead of 9 -- and the pixel shift in the epilogue; see its header.
// conv_sn_small_kernel (3x3 layers with <= 5 output channels: the logits layer): the same with all taps of all classes in one
// 16-column accumulator group.
// conv_igemm_kernel (UAPS_CONV_V1=1): the first, one-tile-per-CTA version, kept for A/B profiling.
#include <cstdio>
#include <cstdlib>
#include "tc_common.cuh"

namespace uaps {
namespace conv {

constexpr int TILE_H = 16, TILE_W = 8, TILE_M = TILE_H * TILE_W;   // 128 pixels = UMMA M
constexpr int THREADS = 128;
constexpr int MAX_STAGES = 8;

struct ConvArgs {
    int B, H, W;
    int cout;            // real output channels (stores are masked beyond it)
    int cout_stride;     // channel pitch of the NHWC output (>= cout)
    int n_tile;          // output channels per CTA, multiple of 16
    int nseg;            // 1 or 2 K segments
    int chunks[2];       // CK-wide channel chunks per segment
    int ks;              // 1 or 3
    int stages;
    int tiles_x, tiles_y;
    int out_nchw_f32;    // 1: write fp32 NCHW (logits), 0: bf16 NHWC
    int num_tiles;       // spatial tiles x n_tiles (persistent kernel)
    int n_tiles;
    int resident;        // 1: this layer's packed weights stay in shared memory for the whole kernel
    int xhalo;           // 1 (resident layers): ONE activation box with an x halo per chunk serves all 9 taps
    const float* bias;   // [>= n_tiles * n_tile] or null
    const unsigned char* w_packed;
    void* out;
    void* out2;          // optional second NHWC output: channels >= split go there (data gradient of a concat conv)
    int split, out2_stride;
    int fold;            // pixel folding factor F (1, 2, 4): the kernel sees [B,H,W/F,F*C] views; only the NCHW / split epilogues care
    int cpp;             // output channels per real pixel in memory (pad16(cout_real))
    int cout_real;
    float act_slope;     // LeakyReLU slope fused into the epilogue (1 = none): inference with BatchNorm folded into the weights
    // BatchNorm batch statistics of the OUTPUT, accumulated by the epilogue (nullable): bn_nrep replicas of
    // [sum[cstride] | sumsq[cstride]] fp64, zeroed by the caller; a CTA adds its per-channel partial sums to replica
    // (blockIdx.x / n_tiles) % bn_nrep -- spreading the same-address atomics, which serialise in L2.
    double* bn_sums;
    int bn_nrep, bn_cstride;
};

// Per-column sums of a 32-lane x 16-column fragment (lane = pixel, v[i] = column i): a recursive-halving butterfly -- at
// every step a lane keeps half of its columns and sends the other half to its partner -- needs 8+4+2+1+1 = 16 shuffles
// instead of the 80 of sixteen independent warp reductions.  Afterwards every lane holds the full sum of column
// (lane >> 1) & 15 (both lanes of a pair hold the same value).
__device__ __forceinline__ float column_sums16(float (&w)[16], int lane) {
#define UAPS_HALVE(N, MASK)                                                             \
    {                                                                                   \
        const bool up = (lane & MASK) != 0;                                             \
        _Pragma("unroll") for (int i = 0; i < N; ++i) {                                 \
            const float send = up ? w[i] : w[i + N];                                    \
            const float keep = up ? w[i + N] : w[i];                                    \
            w[i] = keep + __shfl_xor_sync(0xffffffffu, send, MASK);                     \
        }                                                                               \
    }
    UAPS_HALVE(8, 16) UAPS_HALVE(4, 8) UAPS_HALVE(2, 4) UAPS_HALVE(1, 2)
#undef UAPS_HALVE
    return w[0] + __shfl_xor_sync(0xffffffffu, w[0], 1);
}

using namespace uaps::tc;

// K-major shared-memory matrix descriptor (cute::UMMA::SmemDescriptor): start>>4 | LBO=1 | SBO = 8 rows |
// version 1 | layout type.  Row pitch == swizzle span, so SBO = 8 * span.
template <int CK>
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr) {
    constexpr uint64_t span = CK * 2;                                    // 32 / 64 / 128 bytes
    constexpr uint64_t layout = (CK == 64) ? 2 : (CK == 32 ? 4 : 6);     // SWIZZLE_128B / 64B / 32B
    return (uint64_t)((saddr >> 4) & 0x3FFF) | (1ull << 16) | (((8 * span) >> 4) << 32) | (1ull << 46) | (layout << 61);
}
// same, explicit stride between 8-row groups (x-halo tiles: an image row is TILE_W + 2 pixels apart)
template <int CK>
__device__ __forceinline__ uint64_t make_desc_sbo(uint32_t saddr, uint32_t sbo_bytes) {
    constexpr uint64_t layout = (CK == 64) ? 2 : (CK == 32 ? 4 : 6);
    return (uint64_t)((saddr >> 4) & 0x3FFF) | (1ull << 16) | ((uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32) | (1ull << 46) | (layout << 61);
}
// instruction descriptor (cute::UMMA::InstrDescriptor): D=F32, A=B=BF16, both K-major, N>>3, M>>4
__device__ __forceinline__ uint32_t make_idesc(int n) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(TILE_M >> 4) << 24);
}

template <int CK>
__global__ void __launch_bounds__(THREADS)
conv_igemm_kernel(const __grid_constant__ CUtensorMap map0, const __grid_constant__ CUtensorMap map1,
                  const __grid_constant__ ConvArgs a) {
    constexpr int ROW_BYTES = CK * 2;
    extern __shared__ __align__(1024) unsigned char smem[];
    __shared__ uint64_t full_bar[MAX_STAGES], empty_bar[MAX_STAGES], done_bar;
    __shared__ uint32_t tmem_base_smem;
    grid_dep_launch();

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int halo = a.ks - 1;
    const int a_bytes = (TILE_H + halo) * TILE_W * ROW_BYTES;
    const int b_bytes = a.ks * a.n_tile * ROW_BYTES;
    const int stage_bytes = (a_bytes + b_bytes + 1023) & ~1023;
    const int iters = (a.chunks[0] + (a.nseg > 1 ? a.chunks[1] : 0)) * a.ks;

    // tile coordinates
    int t = blockIdx.x;
    const int tx = t % a.tiles_x; t /= a.tiles_x;
    const int ty = t % a.tiles_y; t /= a.tiles_y;
    const int n_img = t;
    const int x0 = tx * TILE_W, y0 = ty * TILE_H;
    const int n_tile_idx = blockIdx.y;

    uint32_t tmem_cols = 32;
    while ((int)tmem_cols < a.n_tile) tmem_cols <<= 1;

    if (threadIdx.x == 0) {
        for (int s = 0; s < a.stages; ++s) { mbar_init(full_bar + s, 1); mbar_init(empty_bar + s, 1); }
        mbar_init(&done_bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) tmem_alloc(&tmem_base_smem, tmem_cols);
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_d = tmem_base_smem;
    // everything above (barrier init, TMEM allocation) touched no global memory: it overlapped the predecessor's tail
    grid_dep_wait();

    if (warp == 0) {
        if (lane == 0) {
            // ---- TMA producer --------------------------------------------------------------------
            const unsigned char* wsrc = a.w_packed + (size_t)n_tile_idx * iters * b_bytes;
            int it = 0;
            for (int seg = 0; seg < a.nseg; ++seg) {
                const CUtensorMap* map = seg == 0 ? &map0 : &map1;
                for (int ch = 0; ch < a.chunks[seg]; ++ch) {
                    for (int s = 0; s < a.ks; ++s, ++it) {
                        const int st = it % a.stages;
                        mbar_wait(empty_bar + st, ((it / a.stages) & 1) ^ 1);
                        unsigned char* sa = smem + (size_t)st * stage_bytes;
                        mbar_expect_tx(full_bar + st, a_bytes + b_bytes);
                        tma_load_4d(sa, map, ch * CK, x0 + s - halo / 2, y0 - halo / 2, n_img, full_bar + st);
                        bulk_g2s(sa + a_bytes, wsrc + (size_t)it * b_bytes, b_bytes, full_bar + st);
                    }
                }
            }
        }
        __syncwarp();
    } else if (warp == 1) {
        if (lane == 0) {
            // ---- MMA issuer ----------------------------------------------------------------------
            const uint32_t idesc = make_idesc(a.n_tile);
            for (int it = 0; it < iters; ++it) {
                const int st = it % a.stages;
                mbar_wait(full_bar + st, (it / a.stages) & 1);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint32_t sa = smem_u32(smem + (size_t)st * stage_bytes);
                const uint32_t sb = sa + a_bytes;
                for (int r = 0; r < a.ks; ++r) {
#pragma unroll
                    for (int kk = 0; kk < CK / 16; ++kk) {
                        const uint64_t ad = make_desc<CK>(sa + r * (TILE_W * ROW_BYTES) + kk * 32);
                        const uint64_t bd = make_desc<CK>(sb + r * (a.n_tile * ROW_BYTES) + kk * 32);
                        umma_bf16(tmem_d, ad, bd, idesc, (it | r | kk) != 0);
                    }
                }
                umma_commit(empty_bar + st);           // frees the stage when these MMAs have read it
            }
            umma_commit(&done_bar);                    // accumulator complete
        }
        __syncwarp();
    }

    // ---- epilogue: TMEM -> registers -> global ----------------------------------------------------
    mbar_wait(&done_bar, 0);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const int row = warp * 32 + lane;
    const int y = y0 + row / TILE_W, x = x0 + row % TILE_W;
    const bool valid = (y < a.H) && (x < a.W);
    const int n0 = n_tile_idx * a.n_tile;
    for (int j = 0; j < a.n_tile / 16; ++j) {
        float v[16];
        tmem_ld16(tmem_d + ((uint32_t)(warp * 32) << 16) + j * 16, v);
        const int c0 = n0 + j * 16;
        if (a.bias != nullptr) {
#pragma unroll
            for (int i = 0; i < 16; ++i) v[i] += (c0 + i < a.cout) ? __ldg(a.bias + c0 + i) : 0.f;
        }
        if (!valid) continue;
        if (a.out_nchw_f32) {
            float* o = reinterpret_cast<float*>(a.out);
#pragma unroll
            for (int i = 0; i < 16; ++i)
                if (c0 + i < a.cout) o[(((size_t)n_img * a.cout + c0 + i) * a.H + y) * a.W + x] = v[i];
        } else {
            __nv_bfloat16* o = reinterpret_cast<__nv_bfloat16*>(a.out) + (((size_t)n_img * a.H + y) * a.W + x) * a.cout_stride + c0;
            if (c0 + 16 <= a.cout) {
                uint32_t pk[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    __nv_bfloat162 h = __floats2bfloat162_rn(v[2 * i], v[2 * i + 1]);
                    pk[i] = *reinterpret_cast<uint32_t*>(&h);
                }
                uint4* o4 = reinterpret_cast<uint4*>(o);
                o4[0] = make_uint4(pk[0], pk[1], pk[2], pk[3]);
                o4[1] = make_uint4(pk[4], pk[5], pk[6], pk[7]);
            } else {
#pragma unroll
                for (int i = 0; i < 16; ++i)
                    if (c0 + i < a.cout) o[i] = __float2bfloat16_rn(v[i]);
            }
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem_d, tmem_cols);
}

// ---- v2: persistent, warp-specialised, TMEM double-buffered ---------------------------------------------
// One CTA per SM slot loops over output tiles.  warp 0 = TMA producer (runs ahead across tile
// boundaries through the shared-memory ring), warp 1 = MMA issuer (alternates between two TMEM
// accumulators), warps 2-5 = epilogue (drain accumulator i while the MMAs of tile i+1 run).  Layers
// whose packed weights fit in 64 KB keep them resident in shared memory: their stages carry only
// activations, so a tile costs one A box per horizontal tap out of L2 and nothing else.
constexpr int THREADS2 = 192;
constexpr int W_RESIDENT_MAX = 80 * 1024;

__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

template <int CK>
__global__ void __launch_bounds__(THREADS2, 6)
conv_igemm_persistent_kernel(const __grid_constant__ CUtensorMap map0, const __grid_constant__ CUtensorMap map1,
                             const __grid_constant__ ConvArgs a) {
    constexpr int ROW_BYTES = CK * 2;
    extern __shared__ __align__(1024) unsigned char smem[];
    __shared__ uint64_t full_bar[MAX_STAGES], empty_bar[MAX_STAGES], acc_full[2], acc_empty[2], w_bar;
    __shared__ uint32_t tmem_base_smem;
    grid_dep_launch();

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int halo = a.ks - 1;
    const int box_w = a.xhalo ? TILE_W + halo : TILE_W;
    const int a_bytes = (TILE_H + halo) * box_w * ROW_BYTES;
    const int b_bytes = a.ks * a.n_tile * ROW_BYTES;                // the three r-blocks of one (chunk, s)
    const int s_per_it = a.xhalo ? a.ks : 1;                          // horizontal taps served by one stage
    const int iters = (a.chunks[0] + (a.nseg > 1 ? a.chunks[1] : 0)) * a.ks / s_per_it;
    const int w_total = (a.chunks[0] + (a.nseg > 1 ? a.chunks[1] : 0)) * a.ks * b_bytes;
    const int w_region = a.resident ? ((w_total + 1023) & ~1023) : 0;
    const int stage_bytes = (a_bytes + (a.resident ? 0 : b_bytes) + 1023) & ~1023;
    unsigned char* stage0 = smem + w_region;
    // BatchNorm-statistics scratch [epilogue warp][sum | sumsq][n_tile] floats, behind the stages (only when requested)
    float* s_stat = reinterpret_cast<float*>(stage0 + (size_t)a.stages * stage_bytes);
    if (a.bn_sums != nullptr)
        for (int i = threadIdx.x; i < 4 * 2 * a.n_tile; i += THREADS2) s_stat[i] = 0.f;

    uint32_t tmem_cols = 32;
    while ((int)tmem_cols < 2 * a.n_tile) tmem_cols <<= 1;

    if (threadIdx.x == 0) {
        for (int s = 0; s < a.stages; ++s) { mbar_init(full_bar + s, 1); mbar_init(empty_bar + s, 1); }
        for (int b = 0; b < 2; ++b) { mbar_init(acc_full + b, 1); mbar_init(acc_empty + b, 4); }
        mbar_init(&w_bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) tmem_alloc(&tmem_base_smem, tmem_cols);
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_d = tmem_base_smem;
    // everything above (barrier init, TMEM allocation) touched no global memory: it overlapped the predecessor's tail
    grid_dep_wait();

    if (warp == 0) {
        if (lane == 0) {
            // ---- TMA producer ----------------------------------------------------------------------
            if (a.resident) {                                   // n_tiles == 1 whenever the weights are resident
                const int wbytes = w_total;
                mbar_expect_tx(&w_bar, wbytes);
                for (int off = 0; off < wbytes; off += 16384)
                    bulk_g2s(smem + off, a.w_packed + off, min(16384, wbytes - off), &w_bar);
            }
            int itg = 0;
            // tile coordinates advance incrementally (see the epilogue): no div/mod per tile
            int nt = blockIdx.x % a.n_tiles, tq = blockIdx.x / a.n_tiles;
            int tx = tq % a.tiles_x; tq /= a.tiles_x;
            int ty = tq % a.tiles_y;
            int n_img = tq / a.tiles_y;
            const int s_nt = gridDim.x % a.n_tiles;
            int sq = gridDim.x / a.n_tiles;
            const int s_tx = sq % a.tiles_x; sq /= a.tiles_x;
            const int s_ty = sq % a.tiles_y;
            const int s_n = sq / a.tiles_y;
            for (int tile = blockIdx.x; tile < a.num_tiles; tile += gridDim.x,
                     nt += s_nt, tx += (nt >= a.n_tiles), nt -= (nt >= a.n_tiles) ? a.n_tiles : 0,
                     tx += s_tx, ty += (tx >= a.tiles_x), tx -= (tx >= a.tiles_x) ? a.tiles_x : 0,
                     ty += s_ty, n_img += (ty >= a.tiles_y), ty -= (ty >= a.tiles_y) ? a.tiles_y : 0, n_img += s_n) {
                const int x0 = tx * TILE_W, y0 = ty * TILE_H;
                const unsigned char* wsrc = a.w_packed + (size_t)nt * w_total;
                int it = 0;
                for (int seg = 0; seg < a.nseg; ++seg) {
                    const CUtensorMap* map = seg == 0 ? &map0 : &map1;
                    for (int ch = 0; ch < a.chunks[seg]; ++ch) {
                        for (int s = 0; s < a.ks; s += s_per_it, ++it, ++itg) {
                            const int st = itg % a.stages;
                            mbar_wait_relaxed(empty_bar + st, ((itg / a.stages) & 1) ^ 1);
                            unsigned char* sa = stage0 + (size_t)st * stage_bytes;
                            mbar_expect_tx(full_bar + st, a_bytes + (a.resident ? 0 : b_bytes));
                            // xhalo: one box [18][10][CK] starting one pixel left of the tile; else one box per tap s
                            tma_load_4d(sa, map, ch * CK, x0 + (a.xhalo ? 0 : s) - halo / 2, y0 - halo / 2, n_img, full_bar + st);
                            if (!a.resident) bulk_g2s(sa + a_bytes, wsrc + (size_t)it * b_bytes, b_bytes, full_bar + st);
                        }
                    }
                }
            }
        }
        __syncwarp();
    } else if (warp == 1) {
        if (lane == 0) {
            // ---- MMA issuer ------------------------------------------------------------------------
            const uint32_t idesc = make_idesc(a.n_tile);
            if (a.resident) mbar_wait(&w_bar, 0);
            int itg = 0, tcount = 0;
            for (int tile = blockIdx.x; tile < a.num_tiles; tile += gridDim.x, ++tcount) {
                const int buf = tcount & 1;
                mbar_wait(acc_empty + buf, ((tcount >> 1) & 1) ^ 1);        // epilogue has drained this accumulator
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint32_t d = tmem_d + (uint32_t)(buf * a.n_tile);
                for (int it = 0; it < iters; ++it, ++itg) {
                    const int st = itg % a.stages;
                    mbar_wait(full_bar + st, (itg / a.stages) & 1);
                    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                    const uint32_t sa = smem_u32(stage0 + (size_t)st * stage_bytes);
                    for (int s = 0; s < s_per_it; ++s) {
                        // weights of (chunk, s): resident layers index the whole packed image, others their stage
                        const uint32_t sb = a.resident ? smem_u32(smem) + (it * s_per_it + s) * b_bytes : sa + a_bytes;
                        for (int r = 0; r < a.ks; ++r) {
#pragma unroll
                            for (int kk = 0; kk < CK / 16; ++kk) {
                                // xhalo tile rows are (y, x) with x in [0, 10): tap (r, s) starts r rows down, s pixels right,
                                // and consecutive 8-pixel groups are box_w pixels apart
                                const uint64_t ad = make_desc_sbo<CK>(sa + (r * box_w + s) * ROW_BYTES + kk * 32, box_w * ROW_BYTES);
                                const uint64_t bd = make_desc<CK>(sb + r * (a.n_tile * ROW_BYTES) + kk * 32);
                                umma_bf16(d, ad, bd, idesc, (it | s | r | kk) != 0);
                            }
                        }
                    }
                    umma_commit(empty_bar + st);
                }
                umma_commit(acc_full + buf);
            }
        }
        __syncwarp();
    } else {
        // ---- epilogue warps 2..5: TMEM lane quarter = warp % 4 -------------------------------------------
        const int q = warp & 3;
        const int row = q * 32 + lane;
        const int ry = row / TILE_W, rx = row % TILE_W;
        // The small-channel layers are instruction-issue bound (ncu: 315 instructions per epilogue warp per tile, a
        // third of them three integer divisions), so the tile coordinates advance incrementally: mixed-radix step of
        // tile = ((n_img * tiles_y + ty) * tiles_x + tx) * n_tiles + nt by gridDim.x
        int nt = blockIdx.x % a.n_tiles, tq = blockIdx.x / a.n_tiles;
        int tx = tq % a.tiles_x; tq /= a.tiles_x;
        int ty = tq % a.tiles_y;
        int n_img = tq / a.tiles_y;
        const int s_nt = gridDim.x % a.n_tiles;
        int sq = gridDim.x / a.n_tiles;
        const int s_tx = sq % a.tiles_x; sq /= a.tiles_x;
        const int s_ty = sq % a.tiles_y;
        const int s_n = sq / a.tiles_y;
        int tcount = 0;
        for (int tile = blockIdx.x; tile < a.num_tiles; tile += gridDim.x, ++tcount) {
            const int buf = tcount & 1;
            const int y = ty * TILE_H + ry, x = tx * TILE_W + rx;
            const bool valid = (y < a.H) && (x < a.W);
            const int n0 = nt * a.n_tile;
            const int n_cur = n_img;
            // advance to this CTA's next tile
            nt += s_nt; if (nt >= a.n_tiles) { nt -= a.n_tiles; ++tx; }
            tx += s_tx; if (tx >= a.tiles_x) { tx -= a.tiles_x; ++ty; }
            ty += s_ty; if (ty >= a.tiles_y) { ty -= a.tiles_y; ++n_img; }
            n_img += s_n;
            mbar_wait_relaxed(acc_full + buf, (tcount >> 1) & 1);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            for (int j = 0; j < a.n_tile / 16; ++j) {
                float v[16];
                tmem_ld16(tmem_d + ((uint32_t)(q * 32) << 16) + buf * a.n_tile + j * 16, v);
                const int c0 = n0 + j * 16;
                if (a.bias != nullptr) {
                    if (c0 + 16 <= a.cout) {                       // whole group in range: four 16-byte loads
                        const float4* b4 = reinterpret_cast<const float4*>(a.bias + c0);
#pragma unroll
                        for (int i = 0; i < 4; ++i) {
                            const float4 b = __ldg(b4 + i);
                            v[4 * i] += b.x; v[4 * i + 1] += b.y; v[4 * i + 2] += b.z; v[4 * i + 3] += b.w;
                        }
                    } else {                                       // partial group (out_conv: 2 / 4 classes): stop at the last real channel
                        const int nb = a.cout - c0;
#pragma unroll
                        for (int i = 0; i < 16; ++i) { if (i >= nb) break; v[i] += __ldg(a.bias + c0 + i); }
                    }
                }
                if (a.act_slope != 1.f) {
#pragma unroll
                    for (int i = 0; i < 16; ++i) v[i] = v[i] > 0.f ? v[i] : v[i] * a.act_slope;
                }
                if (a.bn_sums != nullptr) {
                    // BatchNorm statistics of this layer's output (UAPS_unet.py:37, 42), from the accumulator while it is in
                    // registers: saves the separate read of the whole output tensor that bn_stats_kernel would do.  The conv
                    // kernels are bound by the tensor core's operand fetch, not by issue slots, so the ~150 extra instructions
                    // per 32 x 16 fragment ride in slack.
                    // (the two quantities one after the other through ONE scratch array: the kernel must stay within 56 registers
                    // for six resident CTAs per SM)
                    const float keep = valid ? 1.f : 0.f;
                    const int col = j * 16 + ((lane >> 1) & 15);
                    float w[16];
#pragma unroll
                    for (int i = 0; i < 16; ++i) w[i] = v[i] * keep;
                    const float cs = column_sums16(w, lane);
                    if ((lane & 1) == 0) s_stat[(q * 2 + 0) * a.n_tile + col] += cs;
#pragma unroll
                    for (int i = 0; i < 16; ++i) w[i] = v[i] * v[i] * keep;
                    const float cq = column_sums16(w, lane);
                    if ((lane & 1) == 0) s_stat[(q * 2 + 1) * a.n_tile + col] += cq;
                }
                if (!valid) continue;
                if (a.out_nchw_f32) {
                    // logits: fp32 NCHW of the REAL image; a folded column block is (sub-pixel, channel)
                    const int sub = a.fold == 1 ? 0 : c0 / a.cpp, cb = a.fold == 1 ? c0 : c0 % a.cpp;
                    const int xr = x * a.fold + sub, Wr = a.W * a.fold;
                    const size_t plane = (size_t)a.H * Wr;
                    float* o = reinterpret_cast<float*>(a.out) + ((size_t)n_cur * a.cout_real + cb) * plane + (size_t)y * Wr + xr;
                    // one pointer walked plane by plane and an early exit after the last real class: the 16 separately
                    // addressed, separately predicated stores this replaces made the 4-class logits layer 85 % slower than
                    // its 16-channel bf16 twin (147 vs 80 us) -- the kernel's time follows the epilogue's instruction count
                    const int nlive = a.cout_real - cb;
#pragma unroll
                    for (int i = 0; i < 16; ++i) { if (i >= nlive) break; *o = v[i]; o += plane; }
                } else {
                    const size_t pix = ((size_t)n_cur * a.H + y) * a.W + x;
                    __nv_bfloat16* o;
                    if (a.out2 != nullptr) {                       // concat data gradient: per real pixel, channels [0,split) | [split,cpp)
                        const int sub = a.fold == 1 ? 0 : c0 / a.cpp, cb = a.fold == 1 ? c0 : c0 % a.cpp, rest = a.cpp - a.split;
                        o = cb < a.split
                            ? reinterpret_cast<__nv_bfloat16*>(a.out) + pix * (size_t)(a.fold * a.split) + sub * a.split + cb
                            : reinterpret_cast<__nv_bfloat16*>(a.out2) + pix * (size_t)(a.fold * rest) + sub * rest + (cb - a.split);
                    } else {
                        o = reinterpret_cast<__nv_bfloat16*>(a.out) + pix * a.cout_stride + c0;
                    }
                    if (c0 + 16 <= a.cout) {
                        uint32_t pk[8];
#pragma unroll
                        for (int i = 0; i < 8; ++i) {
                            __nv_bfloat162 h = __floats2bfloat162_rn(v[2 * i], v[2 * i + 1]);
                            pk[i] = *reinterpret_cast<uint32_t*>(&h);
                        }
                        uint4* o4 = reinterpret_cast<uint4*>(o);
                        o4[0] = make_uint4(pk[0], pk[1], pk[2], pk[3]);
                        o4[1] = make_uint4(pk[4], pk[5], pk[6], pk[7]);
                    } else {
#pragma unroll
                        for (int i = 0; i < 16; ++i)
                            if (c0 + i < a.cout) o[i] = __float2bfloat16_rn(v[i]);
                    }
                }
            }
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            __syncwarp();
            if (lane == 0) mbar_arrive(acc_empty + buf);        // 4 warps -> accumulator free for tile i+2
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem_d, tmem_cols);
    if (a.bn_sums != nullptr && blockIdx.x < (unsigned)a.num_tiles) {
        // this CTA's tiles all have the same output-channel block (the host makes gridDim.x a multiple of n_tiles)
        const int nt = blockIdx.x % a.n_tiles;
        double* rep = a.bn_sums + (size_t)((blockIdx.x / a.n_tiles) % a.bn_nrep) * 2 * a.bn_cstride;
        for (int t = threadIdx.x; t < 2 * a.n_tile; t += THREADS2) {
            const int which = t / a.n_tile, c = t - which * a.n_tile, gc = nt * a.n_tile + c;
            if (gc < a.bn_cstride) {
                const float tot = (s_stat[(0 + which) * a.n_tile + c] + s_stat[(2 + which) * a.n_tile + c]) +
                                  (s_stat[(4 + which) * a.n_tile + c] + s_stat[(6 + which) * a.n_tile + c]);
                atomicAdd(rep + (size_t)which * a.bn_cstride + gc, (double)tot);
            }
        }
    }
}

// ---- v3 ("SN"): the horizontal taps in the N dimension ----------------------------------------------------------
// The kernels above are bound by the tensor core's shared-memory operand fetch: every tcgen05.mma re-reads its 128-row A
// operand, (128 + N) * 32 bytes at 64 B/clk, so a 3x3 conv with N = 16 output channels spends 9 x 72 clocks per 128-pixel
// tile on 9 x 4 clocks of arithmetic (DESIGN.md section 6).  This kernel fetches each A tile three times instead of nine:
//
//     Y_s[p, co] = sum_{r, ci} W[co, ci, r, s] * in[p + (r - 1) rows, ci]         for all three s in ONE MMA:
//                  M = 128 pixels, K = (r, ci), N = (s, co) = 3 * n_co
//     out[p, co] = Y_0[p - 1, co] + Y_1[p, co] + Y_2[p + 1, co]                    in the epilogue
//
// so a tile costs 3 * CK/16 MMAs per channel chunk at (128 + 3 n_co) / 2 clocks each: 264 clocks instead of 648 for
// 16 -> 16 channels, 1920 instead of 3456 for 64 -> 64.  The pixel shift is a warp shuffle: a tile is 4 image rows x 32
// pixels, an epilogue warp owns one row (TMEM lanes 32q..32q+31 = 32 consecutive x) and 16 output channels, and it
// finishes the pixels ONE TO THE LEFT of its lanes: lane l of tile t writes pixel x = 32 t + l - 1 =
// Y_0[lane l - 2] + Y_1[lane l - 1] + Y_2[lane l], two rotating shuffles whose wrapped-around values (lanes 30 / 31 of this
// tile) are exactly what lanes 0 / 1 of the NEXT tile of the band need -- they stay in registers from tile to tile.  A CTA
// sweeps a 4-row band left to right; nothing is computed twice, every output is written once, no pixel waits for data of
// a later tile.  (When W is a multiple of 32 the band's last pixel is finished by lane 31 of the last tile.)
//
//   A operand.  One TMA box {CK, 32 x, 4 + 2 y} per channel chunk: rows (y, x), row pitch = swizzle span; vertical tap r is
//   the same tile read 32 rows further down (atom-aligned).  Rows / columns outside the image are zero-filled.
//   B operand.  All weights resident in shared memory: block (chunk, r) = [3 * n_co rows (s, co)][CK], pre-swizzled.
//   D.  Two accumulators of 3 * n_co fp32 columns.
//   Warps.  0 = TMA producer, 1 = MMA issuer, 2 .. 2 + 4 NG - 1 = epilogue: warp w drains TMEM lane quarter w % 4 (image
//   row w % 4 of the band) of channel group (w - 2) / 4.  The epilogue is ~170 instructions per 32 x 16 fragment and a lone
//   warp issues one every ~9 clocks (ncu), so the 64-channel layers need all sixteen of them to stay under the MMA time.
//   Stores are one contiguous 32 * 32 bytes per warp (NHWC) or 128 bytes per class plane (NCHW logits).
constexpr int SN_TILE_H = 4, SN_TILE_W = 32;

// NG = n_co / 16 output-channel groups = epilogue warps per TMEM lane quarter.  (Fragments of 8 columns -- twice the warps --
// were measured too: 16 -> 16 channels 89 us against 85 us, the epilogue is bound by issue slots, not by latency.)
template <int NG> struct SnCfg {
    static constexpr int EPI_WARPS = 4 * NG;
    static constexpr int THREADS = 64 + 32 * EPI_WARPS;
    // co-resident CTAs: at most 512 / (2 * 48 NG rounded up to a power of two) by their TMEM columns
    static constexpr int MIN_CTAS = NG == 1 ? 4 : (NG == 2 ? 2 : 1);
};

template <int CK, int NG>
__global__ void __launch_bounds__((SnCfg<NG>::THREADS), (SnCfg<NG>::MIN_CTAS))
conv_sn_kernel(const __grid_constant__ CUtensorMap map0, const __grid_constant__ CUtensorMap map1,
               const __grid_constant__ ConvArgs a) {
    constexpr int ROW_BYTES = CK * 2;
    constexpr int A_BYTES = (SN_TILE_H + 2) * SN_TILE_W * ROW_BYTES;          // 6 / 12 / 24 KB, a multiple of 1024
    constexpr int NCO = 16 * NG, N3 = 3 * NCO;
    constexpr int CW = 16;                                                     // columns per epilogue warp
    constexpr int NTHREADS = SnCfg<NG>::THREADS, EPI_WARPS = SnCfg<NG>::EPI_WARPS;
    extern __shared__ __align__(1024) unsigned char smem[];
    __shared__ uint64_t full_bar[MAX_STAGES], empty_bar[MAX_STAGES], acc_full[2], acc_empty[2], w_bar;
    __shared__ uint32_t tmem_base_smem;
    grid_dep_launch();

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int chunks = a.chunks[0] + (a.nseg > 1 ? a.chunks[1] : 0);
    constexpr int RBLOCK = N3 * ROW_BYTES;                                     // weights of one (chunk, r)
    const int w_total = chunks * 3 * RBLOCK;
    const int w_region = (w_total + 1023) & ~1023;
    unsigned char* stage0 = smem + w_region;
    float* s_carry = reinterpret_cast<float*>(stage0 + (size_t)a.stages * A_BYTES);   // [epilogue warp][4][CW]
    float* s_bias = s_carry + EPI_WARPS * 4 * CW;                                      // [n_co]
    float* s_stat = s_bias + NCO;                                                      // [lane quarter][sum | sumsq][n_co]
    for (int i = threadIdx.x; i < NCO; i += NTHREADS) s_bias[i] = (a.bias != nullptr && i < a.cout) ? a.bias[i] : 0.f;
    if (a.bn_sums != nullptr)
        for (int i = threadIdx.x; i < 4 * 2 * NCO; i += NTHREADS) s_stat[i] = 0.f;

    uint32_t tmem_cols = 32;
    while ((int)tmem_cols < 2 * N3) tmem_cols <<= 1;

    if (threadIdx.x == 0) {
        for (int s = 0; s < a.stages; ++s) { mbar_init(full_bar + s, 1); mbar_init(empty_bar + s, 1); }
        for (int b = 0; b < 2; ++b) { mbar_init(acc_full + b, 1); mbar_init(acc_empty + b, EPI_WARPS); }
        mbar_init(&w_bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) tmem_alloc(&tmem_base_smem, tmem_cols);
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_d = tmem_base_smem;
    grid_dep_wait();

    // work unit = (image, band of 4 rows), swept left to right; a.num_tiles = number of units, a.tiles_y = bands per image
    if (warp == 0) {
        if (lane == 0) {
            // ---- TMA producer ----------------------------------------------------------------------
            mbar_expect_tx(&w_bar, w_total);
            for (int off = 0; off < w_total; off += 16384)
                bulk_g2s(smem + off, a.w_packed + off, min(16384, w_total - off), &w_bar);
            int itg = 0;
            for (int unit = blockIdx.x; unit < a.num_tiles; unit += gridDim.x) {
                const int n_img = unit / a.tiles_y, y0 = (unit - n_img * a.tiles_y) * SN_TILE_H;
                for (int tx = 0; tx < a.tiles_x; ++tx) {
                    for (int seg = 0; seg < a.nseg; ++seg) {
                        const CUtensorMap* map = seg == 0 ? &map0 : &map1;
                        for (int ch = 0; ch < a.chunks[seg]; ++ch, ++itg) {
                            const int st = itg % a.stages;
                            mbar_wait_relaxed(empty_bar + st, ((itg / a.stages) & 1) ^ 1);
                            mbar_expect_tx(full_bar + st, A_BYTES);
                            tma_load_4d(stage0 + (size_t)st * A_BYTES, map, ch * CK, tx * SN_TILE_W, y0 - 1, n_img, full_bar + st);
                        }
                    }
                }
            }
        }
        __syncwarp();
    } else if (warp == 1) {
        if (lane == 0) {
            // ---- MMA issuer ------------------------------------------------------------------------
            const uint32_t idesc = make_idesc(N3);
            const uint32_t wbase = smem_u32(smem);
            mbar_wait(&w_bar, 0);
            int itg = 0, tcount = 0;
            for (int unit = blockIdx.x; unit < a.num_tiles; unit += gridDim.x) {
                for (int tx = 0; tx < a.tiles_x; ++tx, ++tcount) {
                    const int buf = tcount & 1;
                    mbar_wait(acc_empty + buf, ((tcount >> 1) & 1) ^ 1);
                    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                    const uint32_t d = tmem_d + (uint32_t)(buf * N3);
                    for (int c = 0; c < chunks; ++c, ++itg) {
                        const int st = itg % a.stages;
                        mbar_wait(full_bar + st, (itg / a.stages) & 1);
                        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                        const uint32_t sa = smem_u32(stage0 + (size_t)st * A_BYTES);
                        const uint32_t sb = wbase + (uint32_t)(c * 3 * RBLOCK);
#pragma unroll
                        for (int r = 0; r < 3; ++r) {
#pragma unroll
                            for (int kk = 0; kk < CK / 16; ++kk) {
                                const uint64_t ad = make_desc<CK>(sa + r * (SN_TILE_W * ROW_BYTES) + kk * 32);
                                const uint64_t bd = make_desc<CK>(sb + r * RBLOCK + kk * 32);
                                umma_bf16(d, ad, bd, idesc, (c | r | kk) != 0);
                            }
                        }
                        umma_commit(empty_bar + st);
                    }
                    umma_commit(acc_full + buf);
                }
            }
        }
        __syncwarp();
    } else {
        // ---- epilogue warps: TMEM lane quarter q = warp % 4 = image row q of the band; columns [c0, c0 + CW) --------
        const int q = warp & 3, g = (warp - 2) >> 2;
        const int c0 = g * CW;
        const size_t plane = (size_t)a.H * a.W;
        const int src2 = (lane + 30) & 31, src1 = (lane + 31) & 31;
        const float m2 = lane < 2 ? 0.f : 1.f, m1 = lane < 1 ? 0.f : 1.f;     // lanes whose neighbours are in the previous tile
        const bool w_full = a.W == a.tiles_x * SN_TILE_W;     // the band's last pixel is lane 31 of the last tile
        // carries of this warp: rows 0 / 1 = Y_0 of lanes 30 / 31, row 2 = Y_1 (+ bias) of lane 31, row 3 = zeros
        float* carry = s_carry + (size_t)(warp - 2) * 4 * CW;
        const float4* cr0 = reinterpret_cast<const float4*>(carry + (lane == 0 ? 0 : CW));       // lane 0: rows 0 + 2; lane 1: rows 1 + 3
        const float4* cr1 = reinterpret_cast<const float4*>(carry + (lane == 0 ? 2 * CW : 3 * CW));
        if (lane < CW) carry[3 * CW + lane] = 0.f;
        const float4* bias4 = reinterpret_cast<const float4*>(s_bias + c0);
        // the epilogue variant is fixed for the launch: one flag instead of a chain of parameter loads and branches per tile
        const bool plain = !a.out_nchw_f32 && a.out2 == nullptr && a.act_slope == 1.f && c0 + CW <= a.cout;
        const bool stats = a.bn_sums != nullptr;
        __syncwarp();

        // one completed pixel per lane: activation, statistics, store
        auto finish = [&](float (&o)[CW], float (&scratch)[CW], bool keep, int n_img, size_t px) {
            if (!plain && a.act_slope != 1.f) {
#pragma unroll
                for (int i = 0; i < CW; ++i) o[i] = o[i] > 0.f ? o[i] : o[i] * a.act_slope;
            }
            if (stats) {
                // BatchNorm statistics of the output (see conv_igemm_persistent_kernel), over the pixels COMPLETED here
                const float kf = keep ? 1.f : 0.f;
                const int col = c0 + ((lane >> 1) & 15);
                const bool owner = (lane & 1) == 0;
#pragma unroll
                for (int i = 0; i < CW; ++i) scratch[i] = o[i] * kf;
                const float cs = column_sums16(scratch, lane);
                if (owner) s_stat[(q * 2 + 0) * NCO + col] += cs;
#pragma unroll
                for (int i = 0; i < CW; ++i) scratch[i] = o[i] * o[i] * kf;
                const float cq = column_sums16(scratch, lane);
                if (owner) s_stat[(q * 2 + 1) * NCO + col] += cq;
            }
            if (!keep) return;
            if (plain) {
                uint32_t pk[CW / 2];
#pragma unroll
                for (int i = 0; i < CW / 2; ++i) {
                    __nv_bfloat162 h = __floats2bfloat162_rn(o[2 * i], o[2 * i + 1]);
                    pk[i] = *reinterpret_cast<uint32_t*>(&h);
                }
                uint4* o4 = reinterpret_cast<uint4*>(reinterpret_cast<__nv_bfloat16*>(a.out) + px * a.cout_stride + c0);
#pragma unroll
                for (int i = 0; i < CW / 8; ++i) o4[i] = make_uint4(pk[4 * i], pk[4 * i + 1], pk[4 * i + 2], pk[4 * i + 3]);
            } else if (a.out_nchw_f32) {
                float* op = reinterpret_cast<float*>(a.out) + ((size_t)n_img * a.cout_real + c0) * plane + (px - (size_t)n_img * plane);
                const int nlive = a.cout_real - c0;
#pragma unroll
                for (int i = 0; i < CW; ++i) { if (i >= nlive) break; *op = o[i]; op += plane; }
            } else {
                __nv_bfloat16* op;
                if (a.out2 != nullptr) {
                    const int rest = a.cpp - a.split;
                    op = c0 < a.split ? reinterpret_cast<__nv_bfloat16*>(a.out) + px * (size_t)a.split + c0
                                      : reinterpret_cast<__nv_bfloat16*>(a.out2) + px * (size_t)rest + (c0 - a.split);
                } else {
                    op = reinterpret_cast<__nv_bfloat16*>(a.out) + px * a.cout_stride + c0;
                }
                if (c0 + CW <= a.cout) {
                    uint32_t pk[CW / 2];
#pragma unroll
                    for (int i = 0; i < CW / 2; ++i) {
                        __nv_bfloat162 h = __floats2bfloat162_rn(o[2 * i], o[2 * i + 1]);
                        pk[i] = *reinterpret_cast<uint32_t*>(&h);
                    }
                    uint4* o4 = reinterpret_cast<uint4*>(op);
#pragma unroll
                    for (int i = 0; i < CW / 8; ++i) o4[i] = make_uint4(pk[4 * i], pk[4 * i + 1], pk[4 * i + 2], pk[4 * i + 3]);
                } else {
#pragma unroll
                    for (int i = 0; i < CW; ++i)
                        if (c0 + i < a.cout) op[i] = __float2bfloat16_rn(o[i]);
                }
            }
        };

        int tcount = 0;
        for (int unit = blockIdx.x; unit < a.num_tiles; unit += gridDim.x) {
            const int n_img = unit / a.tiles_y;
            const int y = (unit - n_img * a.tiles_y) * SN_TILE_H + q;
            const bool yvalid = y < a.H;
            const size_t row_pix = ((size_t)n_img * a.H + y) * a.W;
            for (int tx = 0; tx < a.tiles_x; ++tx, ++tcount) {
                const int buf = tcount & 1;
                const int x = tx * SN_TILE_W + lane - 1;       // the pixel this lane completes
                mbar_wait_relaxed(acc_full + buf, (tcount >> 1) & 1);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                float y0[CW], y1[CW], v[CW];
                const uint32_t tb = tmem_d + ((uint32_t)(q * 32) << 16) + (uint32_t)(buf * N3 + c0);
                tmem_ld16_nowait(tb, y0); tmem_ld16_nowait(tb + NCO, y1); tmem_ld16_nowait(tb + 2 * NCO, v);
                tmem_wait_ld(y0); tmem_ld_fence(y1); tmem_ld_fence(v);
                // the accumulator is in registers: hand it back to the MMA issuer before the arithmetic
                asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
                __syncwarp();
                if (lane == 0) mbar_arrive(acc_empty + buf);
#pragma unroll
                for (int i = 0; i < CW / 4; ++i) {
                    const float4 b = bias4[i];
                    y1[4 * i] += b.x; y1[4 * i + 1] += b.y; y1[4 * i + 2] += b.z; y1[4 * i + 3] += b.w;
                }
#pragma unroll
                for (int i = 0; i < CW; ++i) {
                    const float a0 = __shfl_sync(0xffffffffu, y0[i], src2);
                    const float a1 = __shfl_sync(0xffffffffu, y1[i], src1);
                    v[i] = fmaf(a0, m2, fmaf(a1, m1, v[i]));
                }
                if (tx > 0 && lane < 2) {                      // the neighbours that sit in the previous tile
#pragma unroll
                    for (int i = 0; i < CW / 4; ++i) {
                        const float4 c = cr0[i], d = cr1[i];
                        v[4 * i] += c.x + d.x; v[4 * i + 1] += c.y + d.y; v[4 * i + 2] += c.z + d.z; v[4 * i + 3] += c.w + d.w;
                    }
                }
                __syncwarp();
                if (lane >= 30) {
                    float4* w0 = reinterpret_cast<float4*>(carry + (lane - 30) * CW);
#pragma unroll
                    for (int i = 0; i < CW / 4; ++i) w0[i] = make_float4(y0[4 * i], y0[4 * i + 1], y0[4 * i + 2], y0[4 * i + 3]);
                    if (lane == 31) {
                        float4* w1 = reinterpret_cast<float4*>(carry + 2 * CW);
#pragma unroll
                        for (int i = 0; i < CW / 4; ++i) w1[i] = make_float4(y1[4 * i], y1[4 * i + 1], y1[4 * i + 2], y1[4 * i + 3]);
                    }
                }
                __syncwarp();
                const bool tail = w_full && tx == a.tiles_x - 1;                  // lane 31 also completes its own pixel
                if (tail) {
#pragma unroll
                    for (int i = 0; i < CW; ++i) y1[i] += __shfl_sync(0xffffffffu, y0[i], src1);   // lane 31: Y_0[lane 30] + Y_1 + bias
                }
                finish(v, y0, yvalid && x >= 0 && x < a.W, n_img, row_pix + (size_t)x);
                if (tail) finish(y1, y0, yvalid && lane == 31, n_img, row_pix + (size_t)x + 1);
            }
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem_d, tmem_cols);
    if (a.bn_sums != nullptr && blockIdx.x < (unsigned)a.num_tiles) {
        double* rep = a.bn_sums + (size_t)(blockIdx.x % a.bn_nrep) * 2 * a.bn_cstride;
        for (int t = threadIdx.x; t < 2 * NCO; t += NTHREADS) {
            const int which = t / NCO, c = t - which * NCO;
            if (c < a.bn_cstride) {
                const float tot = (s_stat[(0 + which) * NCO + c] + s_stat[(2 + which) * NCO + c]) +
                                  (s_stat[(4 + which) * NCO + c] + s_stat[(6 + which) * NCO + c]);
                atomicAdd(rep + (size_t)which * a.bn_cstride + c, (double)tot);
            }
        }
    }
}

// ---- v3 for the logits layer: C <= 5 output channels -------------------------------------------------------------
// out_conv (UAPS_unet.py:138-139) has 16 input and 2..4 output channels: with the horizontal taps in N all three taps of all
// classes fit ONE 16-column accumulator group (column s * C + c), so a tile is 3 MMAs of N = 16 and the epilogue reads 16
// TMEM columns and does 2 C shuffles per pixel instead of 48 / 32.  Same tiles, carries and roles as conv_sn_kernel.
// Rows 3 C .. 15 of the packed weight blocks are never written (their accumulator columns are never read).
template <int CK, int C>
__global__ void __launch_bounds__(192, 4)
conv_sn_small_kernel(const __grid_constant__ CUtensorMap map0, const __grid_constant__ CUtensorMap map1,
                     const __grid_constant__ ConvArgs a) {
    constexpr int ROW_BYTES = CK * 2;
    constexpr int A_BYTES = (SN_TILE_H + 2) * SN_TILE_W * ROW_BYTES;
    constexpr int N3 = 16, NTHREADS = 192, CP = 8;                             // CP: carry / bias / statistics row pitch (floats)
    constexpr int RBLOCK = N3 * ROW_BYTES;
    extern __shared__ __align__(1024) unsigned char smem[];
    __shared__ uint64_t full_bar[MAX_STAGES], empty_bar[MAX_STAGES], acc_full[2], acc_empty[2], w_bar;
    __shared__ uint32_t tmem_base_smem;
    grid_dep_launch();

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int chunks = a.chunks[0] + (a.nseg > 1 ? a.chunks[1] : 0);
    const int w_total = chunks * 3 * RBLOCK;
    const int w_region = (w_total + 1023) & ~1023;
    unsigned char* stage0 = smem + w_region;
    float* s_carry = reinterpret_cast<float*>(stage0 + (size_t)a.stages * A_BYTES);   // [epilogue warp][3][CP]
    float* s_bias = s_carry + 4 * 3 * CP;                                              // [CP]
    float* s_stat = s_bias + CP;                                                       // [lane quarter][sum | sumsq][CP]
    if (threadIdx.x < CP) s_bias[threadIdx.x] = (a.bias != nullptr && (int)threadIdx.x < C) ? a.bias[threadIdx.x] : 0.f;
    if (a.bn_sums != nullptr && threadIdx.x < 4 * 2 * CP) s_stat[threadIdx.x] = 0.f;
    constexpr uint32_t tmem_cols = 32;

    if (threadIdx.x == 0) {
        for (int s = 0; s < a.stages; ++s) { mbar_init(full_bar + s, 1); mbar_init(empty_bar + s, 1); }
        for (int b = 0; b < 2; ++b) { mbar_init(acc_full + b, 1); mbar_init(acc_empty + b, 4); }
        mbar_init(&w_bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) tmem_alloc(&tmem_base_smem, tmem_cols);
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_d = tmem_base_smem;
    grid_dep_wait();

    if (warp == 0) {
        if (lane == 0) {
            // ---- TMA producer (as conv_sn_kernel) ----------------------------------------------------
            mbar_expect_tx(&w_bar, w_total);
            for (int off = 0; off < w_total; off += 16384)
                bulk_g2s(smem + off, a.w_packed + off, min(16384, w_total - off), &w_bar);
            int itg = 0;
            for (int unit = blockIdx.x; unit < a.num_tiles; unit += gridDim.x) {
                const int n_img = unit / a.tiles_y, y0 = (unit - n_img * a.tiles_y) * SN_TILE_H;
                for (int tx = 0; tx < a.tiles_x; ++tx) {
                    for (int seg = 0; seg < a.nseg; ++seg) {
                        const CUtensorMap* map = seg == 0 ? &map0 : &map1;
                        for (int ch = 0; ch < a.chunks[seg]; ++ch, ++itg) {
                            const int st = itg % a.stages;
                            mbar_wait_relaxed(empty_bar + st, ((itg / a.stages) & 1) ^ 1);
                            mbar_expect_tx(full_bar + st, A_BYTES);
                            tma_load_4d(stage0 + (size_t)st * A_BYTES, map, ch * CK, tx * SN_TILE_W, y0 - 1, n_img, full_bar + st);
                        }
                    }
                }
            }
        }
        __syncwarp();
    } else if (warp == 1) {
        if (lane == 0) {
            // ---- MMA issuer (as conv_sn_kernel, N = 16) ------------------------------------------------
            const uint32_t idesc = make_idesc(N3);
            const uint32_t wbase = smem_u32(smem);
            mbar_wait(&w_bar, 0);
            int itg = 0, tcount = 0;
            for (int unit = blockIdx.x; unit < a.num_tiles; unit += gridDim.x) {
                for (int tx = 0; tx < a.tiles_x; ++tx, ++tcount) {
                    const int buf = tcount & 1;
                    mbar_wait(acc_empty + buf, ((tcount >> 1) & 1) ^ 1);
                    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                    const uint32_t d = tmem_d + (uint32_t)(buf * N3);
                    for (int c = 0; c < chunks; ++c, ++itg) {
                        const int st = itg % a.stages;
                        mbar_wait(full_bar + st, (itg / a.stages) & 1);
                        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                        const uint32_t sa = smem_u32(stage0 + (size_t)st * A_BYTES);
                        const uint32_t sb = wbase + (uint32_t)(c * 3 * RBLOCK);
#pragma unroll
                        for (int r = 0; r < 3; ++r) {
#pragma unroll
                            for (int kk = 0; kk < CK / 16; ++kk) {
                                const uint64_t ad = make_desc<CK>(sa + r * (SN_TILE_W * ROW_BYTES) + kk * 32);
                                const uint64_t bd = make_desc<CK>(sb + r * RBLOCK + kk * 32);
                                umma_bf16(d, ad, bd, idesc, (c | r | kk) != 0);
                            }
                        }
                        umma_commit(empty_bar + st);
                    }
                    umma_commit(acc_full + buf);
                }
            }
        }
        __syncwarp();
    } else {
        // ---- epilogue warps 2..5: image row q of the band, all C channels ------------------------------------------
        const int q = warp & 3;
        const size_t plane = (size_t)a.H * a.W;
        const int src2 = (lane + 30) & 31, src1 = (lane + 31) & 31;
        const float m2 = lane < 2 ? 0.f : 1.f, m1 = lane < 1 ? 0.f : 1.f;
        const bool w_full = a.W == a.tiles_x * SN_TILE_W;
        float* carry = s_carry + (size_t)(warp - 2) * 3 * CP;      // rows: Y_0 of lane 30, Y_0 of lane 31, Y_1 (+ bias) of lane 31
        float bias[C];
#pragma unroll
        for (int c = 0; c < C; ++c) bias[c] = s_bias[c];
        const bool stats = a.bn_sums != nullptr;
        __syncwarp();

        auto finish = [&](float (&o)[C], bool keep, int n_img, size_t px) {
            if (a.act_slope != 1.f) {
#pragma unroll
                for (int c = 0; c < C; ++c) o[c] = o[c] > 0.f ? o[c] : o[c] * a.act_slope;
            }
            if (stats) {
#pragma unroll
                for (int c = 0; c < C; ++c) {
                    float s1 = keep ? o[c] : 0.f, s2 = s1 * s1;
#pragma unroll
                    for (int sh = 16; sh > 0; sh >>= 1) {
                        s1 += __shfl_xor_sync(0xffffffffu, s1, sh);
                        s2 += __shfl_xor_sync(0xffffffffu, s2, sh);
                    }
                    if (lane == 0) { s_stat[(q * 2 + 0) * CP + c] += s1; s_stat[(q * 2 + 1) * CP + c] += s2; }
                }
            }
            if (!keep) return;
            if (a.out_nchw_f32) {
                float* op = reinterpret_cast<float*>(a.out) + (size_t)n_img * a.cout_real * plane + (px - (size_t)n_img * plane);
#pragma unroll
                for (int c = 0; c < C; ++c) { *op = o[c]; op += plane; }
            } else {
                __nv_bfloat16* op = reinterpret_cast<__nv_bfloat16*>(a.out) + px * a.cout_stride;
#pragma unroll
                for (int c = 0; c < C; ++c) op[c] = __float2bfloat16_rn(o[c]);
            }
        };

        int tcount = 0;
        for (int unit = blockIdx.x; unit < a.num_tiles; unit += gridDim.x) {
            const int n_img = unit / a.tiles_y;
            const int y = (unit - n_img * a.tiles_y) * SN_TILE_H + q;
            const bool yvalid = y < a.H;
            const size_t row_pix = ((size_t)n_img * a.H + y) * a.W;
            for (int tx = 0; tx < a.tiles_x; ++tx, ++tcount) {
                const int buf = tcount & 1;
                const int x = tx * SN_TILE_W + lane - 1;       // the pixel this lane completes
                mbar_wait_relaxed(acc_full + buf, (tcount >> 1) & 1);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                float v[16];
                tmem_ld16(tmem_d + ((uint32_t)(q * 32) << 16) + (uint32_t)(buf * N3), v);
                asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
                __syncwarp();
                if (lane == 0) mbar_arrive(acc_empty + buf);
                float o[C];
#pragma unroll
                for (int c = 0; c < C; ++c) {
                    v[C + c] += bias[c];
                    const float a0 = __shfl_sync(0xffffffffu, v[c], src2);
                    const float a1 = __shfl_sync(0xffffffffu, v[C + c], src1);
                    o[c] = fmaf(a0, m2, fmaf(a1, m1, v[2 * C + c]));
                }
                if (tx > 0 && lane < 2) {
#pragma unroll
                    for (int c = 0; c < C; ++c) o[c] += lane == 0 ? carry[c] + carry[2 * CP + c] : carry[CP + c];
                }
                __syncwarp();
                if (lane >= 30) {
#pragma unroll
                    for (int c = 0; c < C; ++c) {
                        carry[(lane - 30) * CP + c] = v[c];
                        if (lane == 31) carry[2 * CP + c] = v[C + c];
                    }
                }
                __syncwarp();
                const bool tail = w_full && tx == a.tiles_x - 1;
                finish(o, yvalid && x >= 0 && x < a.W, n_img, row_pix + (size_t)x);
                if (tail) {
#pragma unroll
                    for (int c = 0; c < C; ++c) o[c] = __shfl_sync(0xffffffffu, v[c], src1) + v[C + c];
                    finish(o, yvalid && lane == 31, n_img, row_pix + (size_t)x + 1);
                }
            }
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem_d, tmem_cols);
    if (a.bn_sums != nullptr && blockIdx.x < (unsigned)a.num_tiles && threadIdx.x < 2 * C) {
        const int which = threadIdx.x / C, c = threadIdx.x - which * C;
        double* rep = a.bn_sums + (size_t)(blockIdx.x % a.bn_nrep) * 2 * a.bn_cstride;
        const float tot = (s_stat[(0 + which) * CP + c] + s_stat[(2 + which) * CP + c]) +
                          (s_stat[(4 + which) * CP + c] + s_stat[(6 + which) * CP + c]);
        atomicAdd(rep + (size_t)which * a.bn_cstride + c, (double)tot);
    }
}

// ---- weight packing: torch [Cout][Cin][ks][ks] fp32 -> pre-swizzled bf16 stage images -----------------
// dst block (nt, it = ((seg, chunk), s), r) is [n_tile][CK] bf16; 16-byte chunk j of row n is stored at
// chunk (j ^ swz(n)) -- Swizzle<3|2|1,4,3> on the byte address, the pattern TMA / UMMA use.
struct PackArgs {
    const float* w; unsigned char* dst;
    int cout_real, cin_total_real, ks, n_tile, n_tiles, ck, nseg;
    int seg_real[2];     // channels of each K segment that have weights
    int seg_mem[2];      // channels per pixel of each segment's tensor in memory (multiple of 16; zeros beyond seg_real)
    int cout_mem;        // output channels per pixel in memory (pad16)
    int fold;            // F: the virtual conv works on [.., W/F, F*C] views
    int transpose;       // 1: logical W'[co][ci][r][s] = W[ci][co][ks-1-r][ks-1-s] (data-gradient conv)
    int sn;              // 1: layout of conv_sn_kernel: block (chunk, r) = [3 * n_tile rows (s, co)][CK]; 2: conv_sn_small_kernel
};
// logical (unfolded) weight of the convolution being packed
__device__ __forceinline__ float logical_w(const PackArgs& p, int co, int ci, int r, int s) {
    if (!p.transpose) return p.w[(((size_t)co * p.cin_total_real + ci) * p.ks + r) * p.ks + s];
    return p.w[(((size_t)ci * p.cout_real + co) * p.ks + (p.ks - 1 - r)) * p.ks + (p.ks - 1 - s)];
}
// Pixel folding: F horizontally adjacent pixels of a small-channel tensor are viewed as one pixel with F*C
// channels (same memory).  The virtual conv has Cin' = F*Cin, Cout' = F*Cout and three horizontal taps dj over
// folded pixels; virtual weight [(b,co)][(a,ci)][r][dj] = W[co][ci][r][s] with s = (dj-1)*F + a - b + 1 when
// that is a real tap, else 0.  F x more MACs (free: these layers are bandwidth bound), F x wider TMA rows.
__device__ __forceinline__ void pack_weights_body(const PackArgs& p, long long first, long long stride);

__global__ void pack_weights_kernel(PackArgs p) {
    grid_dep_launch();
    grid_dep_wait();
    pack_weights_body(p, (long long)blockIdx.x * blockDim.x + threadIdx.x, (long long)gridDim.x * blockDim.x);
}

// Every layer of the network in ONE launch (uaps_conv_pack_run): a device table holds one PackArgs per (layer, layout)
// plus the first block of each job; a block finds its job by scanning the (<= a few hundred) starts.  Replaces the 124
// launches of 4-5 us that packing weights layer by layer costs per training iteration.
struct PackJob { PackArgs args; int first_block; int n_blocks; };
__global__ void pack_weights_batched_kernel(const PackJob* __restrict__ jobs, int n_jobs) {
    grid_dep_launch();
    grid_dep_wait();
    __shared__ int s_job;
    if (threadIdx.x == 0) {
        int lo = 0, hi = n_jobs - 1;                      // last job whose first_block <= blockIdx.x
        while (lo < hi) {
            const int mid = (lo + hi + 1) >> 1;
            if (jobs[mid].first_block <= (int)blockIdx.x) lo = mid; else hi = mid - 1;
        }
        s_job = lo;
    }
    __syncthreads();
    const PackJob& j = jobs[s_job];
    pack_weights_body(j.args, (long long)((int)blockIdx.x - j.first_block) * blockDim.x + threadIdx.x,
                      (long long)j.n_blocks * blockDim.x);
}

__device__ __forceinline__ void pack_weights_body(const PackArgs& p, long long first, long long stride) {
    const int F = p.fold;
    const int chunks_per_row = p.ck / 8;
    const int chunks0 = F * p.seg_mem[0] / p.ck, chunks1 = p.nseg > 1 ? F * p.seg_mem[1] / p.ck : 0;
    const int iters = (chunks0 + chunks1) * p.ks;
    const int cout_v = F * p.cout_mem;
    const long long total = (long long)p.n_tiles * iters * p.ks * p.n_tile * chunks_per_row;
    for (long long idx = first; idx < total; idx += stride) {
        long long t = idx;
        const int j = t % chunks_per_row; t /= chunks_per_row;
        const int n = t % p.n_tile; t /= p.n_tile;
        const int r = t % p.ks; t /= p.ks;
        const int it = t % iters; t /= iters;
        const int nt = (int)t;
        const int dj = it % p.ks;
        int ch = it / p.ks, seg = 0;
        if (ch >= chunks0) { ch -= chunks0; seg = 1; }
        const int cov = nt * p.n_tile + n;                             // virtual output channel = (b, co)
        const int b = cov / p.cout_mem, co = cov % p.cout_mem;
        const int span_rows = 128 / (p.ck * 2);                         // rows per 128 bytes: 1 / 2 / 4
        const int swz = (n / span_rows) % chunks_per_row;               // bits [7,7+B) of the byte address
        __nv_bfloat16 vals[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            const int clv = ch * p.ck + j * 8 + e;                      // virtual channel inside the segment = (a, cl)
            const int a = clv / p.seg_mem[seg], cl = clv % p.seg_mem[seg];
            const int s = p.ks == 3 ? (dj - 1) * F + a - b + 1 : (a == b ? 0 : -1);
            float v = 0.f;
            if (cov < cout_v && co < p.cout_real && cl < p.seg_real[seg] && s >= 0 && s < p.ks)
                v = logical_w(p, co, (seg == 0 ? 0 : p.seg_real[0]) + cl, r, s);
            vals[e] = __float2bfloat16_rn(v);
        }
        size_t off;
        if (p.sn == 2) {                                                // conv_sn_small_kernel: 16-row blocks, row s * C + co
            if (n >= p.cout_real) continue;
            const int np = dj * p.cout_real + n;
            const int swz_sn = (np / span_rows) % chunks_per_row;
            off = ((size_t)(it / p.ks) * p.ks + r) * (size_t)16 * (p.ck * 2) + (size_t)np * (p.ck * 2) + (size_t)((j ^ swz_sn) * 16);
        } else if (p.sn) {                                              // (n_tiles = 1, F = 1, ks = 3)
            const int np = dj * p.n_tile + n;                           // row (s, co) of the block of (chunk, r)
            const int swz_sn = (np / span_rows) % chunks_per_row;
            off = ((size_t)(it / p.ks) * p.ks + r) * (size_t)(p.ks * p.n_tile) * (p.ck * 2) + (size_t)np * (p.ck * 2) +
                  (size_t)((j ^ swz_sn) * 16);
        } else {
            const size_t block = (((size_t)nt * iters + it) * p.ks + r) * p.n_tile * (p.ck * 2);
            off = block + (size_t)n * (p.ck * 2) + (size_t)((j ^ swz) * 16);
        }
        *reinterpret_cast<uint4*>(p.dst + off) = *reinterpret_cast<const uint4*>(vals);
    }
}

inline int pick_ck(int c) { return c % 64 == 0 ? 64 : (c % 32 == 0 ? 32 : 16); }
inline int pick_n_tile(int cout) {
    const int padded = (cout + 15) / 16 * 16;
    return padded <= 128 ? padded : 128;
}

}  // namespace conv
}  // namespace uaps

using namespace uaps;
using namespace uaps::conv;

namespace {
struct Plan {
    int ck, n_tile, n_tiles, seg_pad[2], chunks[2], nseg, iters;
    int sn;              // 1: conv_sn_kernel (horizontal taps in N) and its weight layout; 2: conv_sn_small_kernel (cout <= 5)
    size_t packed_bytes;
};
// conv_sn_kernel takes 3x3 layers with <= 64 (padded) output channels whose packed weights stay resident next to two
// activation stages: every 16- / 32- / 64-channel layer of UNet_UAPS and the data gradients that produce them.
// UAPS_CONV_SN=0 keeps those layers on conv_igemm_persistent_kernel (A/B profiling).
constexpr size_t SN_W_MAX = 150 * 1024;
inline bool sn_enabled() {
    static const bool on = [] {
        const char* e = getenv("UAPS_CONV_SN");
        return (e == nullptr || atoi(e) != 0) && getenv("UAPS_CONV_V1") == nullptr;
    }();
    return on;
}
// cin2 == 0: single segment.  Channels are zero-padded up to a multiple of 16 inside a segment; with pixel folding
// (fold = F > 1) the plan is made for the virtual conv on the [.., W/F, F*C] views.
int make_plan(int cout, int cin1, int cin2, int ks, int fold, Plan* pl) {
    if (cout <= 0 || cin1 <= 0 || cin2 < 0 || (ks != 1 && ks != 3) || (fold != 1 && fold != 2 && fold != 4)) return UAPS_EINVAL;
    pl->nseg = cin2 > 0 ? 2 : 1;
    pl->seg_pad[0] = fold * ((cin1 + 15) / 16 * 16);
    pl->seg_pad[1] = fold * ((cin2 + 15) / 16 * 16);
    int ck = pick_ck(pl->seg_pad[0]);
    if (pl->nseg > 1) { const int ck2 = pick_ck(pl->seg_pad[1]); if (ck2 < ck) ck = ck2; }
    pl->ck = ck;
    pl->chunks[0] = pl->seg_pad[0] / ck;
    pl->chunks[1] = pl->nseg > 1 ? pl->seg_pad[1] / ck : 0;
    const int cout_v = fold > 1 ? fold * ((cout + 15) / 16 * 16) : cout;
    pl->n_tile = pick_n_tile(cout_v);
    pl->n_tiles = (cout_v + pl->n_tile - 1) / pl->n_tile;
    pl->iters = (pl->chunks[0] + pl->chunks[1]) * ks;
    pl->packed_bytes = (size_t)pl->n_tiles * pl->iters * ks * pl->n_tile * ck * 2;
    // ... and only where it wins (measured per layer, B = 64, profiles/r02_conv_sn_layers.txt): its epilogue reads three
    // accumulator columns per output and is bound by issue slots at ~170 instructions per 32 x 16 fragment, so it pays when
    // there is enough K behind every output column: input channels >= 2 x output channels, or >= 64.
    const int cin_pad = pl->seg_pad[0] + (pl->nseg > 1 ? pl->seg_pad[1] : 0);
    static const bool sn_all = [] { const char* e = getenv("UAPS_CONV_SN"); return e != nullptr && atoi(e) == 2; }();   // 2: every eligible layer
    pl->sn = (sn_enabled() && ks == 3 && fold == 1 && pl->n_tiles == 1 && pl->n_tile <= 64 && pl->packed_bytes <= SN_W_MAX &&
              (sn_all || cin_pad >= 2 * pl->n_tile || cin_pad >= 64)) ? 1 : 0;
    if (sn_enabled() && ks == 3 && fold == 1 && cout <= 5 && pl->packed_bytes <= SN_W_MAX) pl->sn = 2;    // the logits layer
    return UAPS_OK;
}

// cuTensorMapEncodeTiled is a driver-API symbol; it is resolved through the runtime at first use so the
// library has no link-time dependency on libcuda (it must still dlopen on a box without a driver).
using EncodeTiledFn = CUresult (*)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                   const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                   CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn encode_tiled_fn() {
    static const EncodeTiledFn fn = [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
            q != cudaDriverEntryPointSuccess)
            p = nullptr;
        return reinterpret_cast<EncodeTiledFn>(p);
    }();
    return fn;
}

int encode_map(CUtensorMap* map, const void* ptr, int B, int H, int W, int C, int ck, int box_h, int box_w = TILE_W) {
    EncodeTiledFn encode = encode_tiled_fn();
    if (encode == nullptr) return UAPS_ENODEV;
    cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)B};
    cuuint64_t strides[3] = {(cuuint64_t)C * 2, (cuuint64_t)W * C * 2, (cuuint64_t)H * W * C * 2};
    cuuint32_t box[4] = {(cuuint32_t)ck, (cuuint32_t)box_w, (cuuint32_t)box_h, 1};
    cuuint32_t estr[4] = {1, 1, 1, 1};
    const CUtensorMapSwizzle sw = ck == 64 ? CU_TENSOR_MAP_SWIZZLE_128B : (ck == 32 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B);
    CUresult r = encode(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(ptr), dims, strides, box, estr,
                                        CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? UAPS_OK : UAPS_EINVAL;
}
}  // namespace

UAPS_API size_t uaps_conv_packed_bytes(int cout, int cin1, int cin2, int ks, int fold) {
    Plan pl;
    if (make_plan(cout, cin1, cin2, ks, fold, &pl) != UAPS_OK) return 0;
    return pl.packed_bytes;
}

namespace {
int make_pack_args(const float* w, void* w_packed, int cout, int cin1, int cin2, int ks, int transpose, int fold, PackArgs* out,
                   int* grid) {
    Plan pl;
    int rc = make_plan(cout, cin1, cin2, ks, fold, &pl);
    if (rc != UAPS_OK) return rc;
    if (w == nullptr || w_packed == nullptr) return UAPS_EINVAL;
    if (!aligned_to(w_packed, 16)) return UAPS_EALIGN;
    PackArgs p{};
    p.w = w; p.dst = reinterpret_cast<unsigned char*>(w_packed);
    p.cout_real = cout; p.cin_total_real = cin1 + cin2; p.ks = ks; p.n_tile = pl.n_tile; p.n_tiles = pl.n_tiles; p.ck = pl.ck;
    p.nseg = pl.nseg; p.seg_real[0] = cin1; p.seg_real[1] = cin2;
    p.seg_mem[0] = (cin1 + 15) / 16 * 16; p.seg_mem[1] = (cin2 + 15) / 16 * 16;
    // unfolded outputs are addressed by real channel (stores beyond cout are masked); folded ones per padded pixel
    p.cout_mem = fold > 1 ? (cout + 15) / 16 * 16 : pl.n_tiles * pl.n_tile;
    p.fold = fold; p.transpose = transpose; p.sn = pl.sn;
    const long long total = (long long)pl.packed_bytes / 16;
    *grid = (int)((total + 255) / 256 < 1184 ? (total + 255) / 256 : 1184);
    *out = p;
    return UAPS_OK;
}
}  // namespace

UAPS_API int uaps_conv_pack_weights(const float* w, void* w_packed, int cout, int cin1, int cin2, int ks, int transpose,
                                    int fold, cudaStream_t stream) {
    PackArgs p{};
    int grid = 0;
    const int rc = make_pack_args(w, w_packed, cout, cin1, cin2, ks, transpose, fold, &p, &grid);
    if (rc != UAPS_OK) return rc;
    UAPS_LAUNCH(pack_weights_kernel, dim3(grid), dim3(256), 0, stream, p);
    UAPS_LAUNCH_CHECK();
    return UAPS_OK;
}

// ---- all layers in one launch -------------------------------------------------------------------------------
// uaps_conv_pack_plan fills a HOST table (n_jobs records of uaps_conv_pack_job_bytes() bytes) from the job list; the caller
// copies it to device memory once (the pointers in it are the parameters' and the packed buffers' device addresses, which
// must stay fixed -- true for parameters living in a flat buffer); uaps_conv_pack_run then re-packs every layer from the
// current parameter values with a single launch, e.g. at the top of every training iteration.
UAPS_API size_t uaps_conv_pack_job_bytes(void) { return sizeof(PackJob); }

UAPS_API int uaps_conv_pack_plan(const UapsPackJob* jobs, int n_jobs, void* table_host, int* total_blocks) {
    if (jobs == nullptr || table_host == nullptr || total_blocks == nullptr || n_jobs <= 0) return UAPS_EINVAL;
    PackJob* out = reinterpret_cast<PackJob*>(table_host);
    int next = 0;
    for (int i = 0; i < n_jobs; ++i) {
        int grid = 0;
        const int rc = make_pack_args(jobs[i].w, jobs[i].w_packed, jobs[i].cout, jobs[i].cin1, jobs[i].cin2, jobs[i].ks,
                                      jobs[i].transpose, jobs[i].fold, &out[i].args, &grid);
        if (rc != UAPS_OK) return rc;
        if (grid > 64) grid = 64;                      // many small jobs share the machine: cap one job's blocks
        out[i].first_block = next;
        out[i].n_blocks = grid;
        next += grid;
    }
    *total_blocks = next;
    return UAPS_OK;
}

UAPS_API int uaps_conv_pack_run(const void* table_dev, int n_jobs, int total_blocks, cudaStream_t stream) {
    if (table_dev == nullptr || n_jobs <= 0 || total_blocks <= 0) return UAPS_EINVAL;
    if (!aligned_to(table_dev, 8)) return UAPS_EALIGN;
    UAPS_LAUNCH(pack_weights_batched_kernel, dim3(total_blocks), dim3(256), 0, stream, reinterpret_cast<const PackJob*>(table_dev),
                n_jobs);
    UAPS_LAUNCH_CHECK();
    return UAPS_OK;
}

UAPS_API int uaps_conv_fprop_act(const void* x1, int c1_stride, const void* x2, int c2_stride, const void* w_packed,
                                 const float* bias, void* out, int out_c_stride, int out_nchw_f32, int B, int H, int W,
                                 int cin1, int cin2, int cout, int ks, void* out2, int out2_c_stride, int split,
                                 int fold, float leaky_slope, cudaStream_t stream);
UAPS_API int uaps_conv_fprop_bn(const void* x1, int c1_stride, const void* x2, int c2_stride, const void* w_packed,
                                const float* bias, void* out, int out_c_stride, int B, int H, int W, int cin1, int cin2,
                                int cout, int ks, double* bn_sums, int bn_nrep, cudaStream_t stream);

UAPS_API int uaps_conv_fprop(const void* x1, int c1_stride, const void* x2, int c2_stride, const void* w_packed,
                             const float* bias, void* out, int out_c_stride, int out_nchw_f32, int B, int H, int W,
                             int cin1, int cin2, int cout, int ks, void* out2, int out2_c_stride, int split,
                             int fold, cudaStream_t stream) {
    return uaps_conv_fprop_act(x1, c1_stride, x2, c2_stride, w_packed, bias, out, out_c_stride, out_nchw_f32, B, H, W, cin1, cin2,
                               cout, ks, out2, out2_c_stride, split, fold, 1.0f, stream);
}

// Same with y = leaky_relu(conv(x) + bias, leaky_slope) applied in the epilogue (leaky_slope = 1: identity).  With BatchNorm's
// running statistics folded into the weights and bias this is a whole eval-mode ConvBlock layer (UAPS_unet.py:36-43) in one kernel.
namespace {
int conv_fprop_impl(const void* x1, int c1_stride, const void* x2, int c2_stride, const void* w_packed, const float* bias,
                    void* out, int out_c_stride, int out_nchw_f32, int B, int H, int W, int cin1, int cin2, int cout, int ks,
                    void* out2, int out2_c_stride, int split, int fold, float leaky_slope, double* bn_sums, int bn_nrep,
                    cudaStream_t stream);
}

UAPS_API int uaps_conv_fprop_act(const void* x1, int c1_stride, const void* x2, int c2_stride, const void* w_packed,
                                 const float* bias, void* out, int out_c_stride, int out_nchw_f32, int B, int H, int W,
                                 int cin1, int cin2, int cout, int ks, void* out2, int out2_c_stride, int split,
                                 int fold, float leaky_slope, cudaStream_t stream) {
    return conv_fprop_impl(x1, c1_stride, x2, c2_stride, w_packed, bias, out, out_c_stride, out_nchw_f32, B, H, W, cin1, cin2, cout,
                           ks, out2, out2_c_stride, split, fold, leaky_slope, nullptr, 0, stream);
}

// conv + bias -> bf16 NHWC as uaps_conv_fprop, and the BatchNorm batch statistics of that output in the same kernel:
// bn_sums = bn_nrep replicas of [sum[out_c_stride] | sumsq[out_c_stride]] doubles, zeroed by the caller; the statistics of the
// whole output are the sums over the replicas (uaps_bn_act_nhwc takes them as they are).
UAPS_API int uaps_conv_fprop_bn(const void* x1, int c1_stride, const void* x2, int c2_stride, const void* w_packed,
                                const float* bias, void* out, int out_c_stride, int B, int H, int W, int cin1, int cin2,
                                int cout, int ks, double* bn_sums, int bn_nrep, cudaStream_t stream) {
    if (bn_sums == nullptr || bn_nrep < 1 || bn_nrep > 64 || !aligned_to(bn_sums, 8)) return UAPS_EINVAL;
    return conv_fprop_impl(x1, c1_stride, x2, c2_stride, w_packed, bias, out, out_c_stride, 0, B, H, W, cin1, cin2, cout, ks, nullptr,
                           0, 0, 1, 1.0f, bn_sums, bn_nrep, stream);
}

namespace {
int conv_fprop_impl(const void* x1, int c1_stride, const void* x2, int c2_stride, const void* w_packed, const float* bias,
                    void* out, int out_c_stride, int out_nchw_f32, int B, int H, int W, int cin1, int cin2, int cout, int ks,
                    void* out2, int out2_c_stride, int split, int fold, float leaky_slope, double* bn_sums, int bn_nrep,
                    cudaStream_t stream) {
    // fold = F > 1: run the virtual convolution on the [B, H, W/F, F*C] views of the same tensors.  Requires the
    // tensors' channel pitch to equal their padded channel count (so F pixels are contiguous) and W % F == 0.
    Plan pl;
    const int cout_real = cout, cpp = (cout + 15) / 16 * 16;
    if (fold > 1) {
        if (W % fold != 0 || c1_stride != (cin1 + 15) / 16 * 16 || (cin2 > 0 && c2_stride != (cin2 + 15) / 16 * 16)) return UAPS_ERANGE;
        if (!out_nchw_f32 && out2 == nullptr && out_c_stride != cpp) return UAPS_ERANGE;
    }
    int rc = make_plan(cout, cin1, cin2, ks, fold, &pl);
    if (rc == UAPS_OK && fold > 1) {                 // from here on: virtual sizes
        W /= fold; c1_stride *= fold; c2_stride *= fold; out_c_stride *= fold;
        cin1 = c1_stride; cin2 = cin2 > 0 ? c2_stride : 0; cout = fold * cpp;
    }
    if (rc != UAPS_OK) return rc;
    if (x1 == nullptr || w_packed == nullptr || out == nullptr || B <= 0 || H <= 0 || W <= 0) return UAPS_EINVAL;
    if (cin2 > 0 && x2 == nullptr) return UAPS_EINVAL;
    // the activation tensors must physically hold the zero-padded channel count (c*_stride), 16-byte aligned rows
    if (c1_stride < pl.seg_pad[0] || (c1_stride % 8) != 0 || (cin2 > 0 && (c2_stride < pl.seg_pad[1] || (c2_stride % 8) != 0)))
        return UAPS_ERANGE;
    if (!aligned_to(x1, 16) || (x2 && !aligned_to(x2, 16)) || !aligned_to(out, 16) || !aligned_to(w_packed, 16) ||
        (bias && !aligned_to(bias, 16)))
        return UAPS_EALIGN;
    if (!out_nchw_f32 && (out_c_stride < (out2 != nullptr ? split : cout) || (out_c_stride % 8) != 0)) return UAPS_ERANGE;
    if (out2 != nullptr && out2_c_stride < cpp - split) return UAPS_ERANGE;

    ConvArgs a{};
    a.B = B; a.H = H; a.W = W; a.cout = cout; a.cout_stride = out_c_stride; a.n_tile = pl.n_tile; a.nseg = pl.nseg;
    a.chunks[0] = pl.chunks[0]; a.chunks[1] = pl.chunks[1]; a.ks = ks;
    a.tiles_x = (W + TILE_W - 1) / TILE_W; a.tiles_y = (H + TILE_H - 1) / TILE_H;
    a.out_nchw_f32 = out_nchw_f32; a.bias = bias; a.w_packed = reinterpret_cast<const unsigned char*>(w_packed); a.out = out;
    a.out2 = out2; a.split = split; a.out2_stride = out2_c_stride;
    a.fold = fold; a.cpp = (fold > 1 || out2 != nullptr) ? cpp : cout; a.cout_real = cout_real;
    a.act_slope = leaky_slope;
    a.bn_sums = bn_sums; a.bn_nrep = bn_nrep; a.bn_cstride = out_c_stride;
    if (bn_sums != nullptr && (getenv("UAPS_CONV_V1") != nullptr || out_nchw_f32 || out2 != nullptr || fold != 1)) return UAPS_EINVAL;
    if (leaky_slope != 1.0f && getenv("UAPS_CONV_V1") != nullptr) return UAPS_EINVAL;      // the v1 kernel has no activation epilogue
    if (out2 != nullptr && (out_nchw_f32 || (split % 16) != 0 || split <= 0 || split >= cpp || (out2_c_stride % 8) != 0 ||
                            !aligned_to(out2, 16) || getenv("UAPS_CONV_V1") != nullptr))
        return UAPS_EINVAL;
    const int row_bytes = pl.ck * 2;
    const int a_bytes = (TILE_H + ks - 1) * TILE_W * row_bytes, b_bytes = ks * pl.n_tile * row_bytes;
    a.n_tiles = pl.n_tiles;
    a.num_tiles = a.tiles_x * a.tiles_y * B * pl.n_tiles;

    if (pl.sn) {
        // conv_sn_kernel: work unit = (image, band of 4 rows); resident weights; as many activation stages as fit the CTA's
        // share of shared memory (the number of co-resident CTAs is set by their TMEM columns, at most 4)
        a.tiles_x = (W + SN_TILE_W - 1) / SN_TILE_W; a.tiles_y = (H + SN_TILE_H - 1) / SN_TILE_H;
        a.num_tiles = a.tiles_y * B; a.n_tiles = 1; a.resident = 1; a.xhalo = 0;
        CUtensorMap m0, m1;
        rc = encode_map(&m0, x1, B, H, W, c1_stride, pl.ck, SN_TILE_H + 2, SN_TILE_W);
        if (rc != UAPS_OK) return rc;
        rc = encode_map(&m1, cin2 > 0 ? x2 : x1, B, H, W, cin2 > 0 ? c2_stride : c1_stride, pl.ck, SN_TILE_H + 2, SN_TILE_W);
        if (rc != UAPS_OK) return rc;
        if (pl.sn == 2) {
            if (out2 != nullptr) return UAPS_EINVAL;                   // (a split output needs >= 32 channels)
            const size_t w_region = ((size_t)(pl.chunks[0] + pl.chunks[1]) * 3 * 16 * row_bytes + 1023) & ~(size_t)1023;
            const size_t stage_bytes = (size_t)(SN_TILE_H + 2) * SN_TILE_W * row_bytes;
            const size_t extra = (size_t)(4 * 3 * 8 + 8 + 4 * 2 * 8) * sizeof(float) + 1024;
            int per_sm = 4, stages = 6;
            while (stages > 2 && w_region + stages * stage_bytes + extra + 2048 > (size_t)(227 * 1024) / per_sm) --stages;
            while (per_sm > 1 && w_region + stages * stage_bytes + extra + 2048 > (size_t)(227 * 1024) / per_sm) --per_sm;
            a.stages = stages;
            const size_t smem = w_region + stages * stage_bytes + extra;
            if (smem > 227 * 1024) return UAPS_ERANGE;
            long long gridx = (long long)device_info().sm_count * per_sm;
            if (gridx > a.num_tiles) gridx = a.num_tiles;
            if (getenv("UAPS_CONV_DEBUG") != nullptr)
                fprintf(stderr, "conv_sn_small<%d,%d>: per_sm %d stages %d smem %zu units %d\n", pl.ck, cout_real, per_sm, stages,
                        smem, a.num_tiles);
            cudaError_t e;
#define UAPS_CONV_LAUNCH4(CKV, CV)                                                                                          \
            e = cudaFuncSetAttribute(conv_sn_small_kernel<CKV, CV>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);   \
            if (e != cudaSuccess) return (int)e;                                                                            \
            UAPS_LAUNCH((conv_sn_small_kernel<CKV, CV>), dim3((unsigned)gridx), dim3(192), smem, stream, m0, m1, a);
#define UAPS_CONV_LAUNCH4_C(CKV)                                                                   \
            switch (cout_real) {                                                                   \
                case 1: { UAPS_CONV_LAUNCH4(CKV, 1) } break;                                       \
                case 2: { UAPS_CONV_LAUNCH4(CKV, 2) } break;                                       \
                case 3: { UAPS_CONV_LAUNCH4(CKV, 3) } break;                                       \
                case 4: { UAPS_CONV_LAUNCH4(CKV, 4) } break;                                       \
                default: { UAPS_CONV_LAUNCH4(CKV, 5) } break;                                      \
            }
            if (pl.ck == 64) { UAPS_CONV_LAUNCH4_C(64) } else if (pl.ck == 32) { UAPS_CONV_LAUNCH4_C(32) } else { UAPS_CONV_LAUNCH4_C(16) }
#undef UAPS_CONV_LAUNCH4_C
#undef UAPS_CONV_LAUNCH4
            UAPS_LAUNCH_CHECK();
            return UAPS_OK;
        }
        const int ng = pl.n_tile / 16;                      // epilogue warp groups (16 output channels each)
        const int n3 = 3 * pl.n_tile;
        int tmem_cols = 32;
        while (tmem_cols < 2 * n3) tmem_cols <<= 1;
        static const int cap_sn = [] { const char* e = getenv("UAPS_CONV_SN_CTAS_PER_SM"); return e ? atoi(e) : 4; }();
        int per_sm = 512 / tmem_cols;
        if (per_sm > cap_sn) per_sm = cap_sn;
        if (per_sm < 1) per_sm = 1;
        const size_t w_region = (pl.packed_bytes + 1023) & ~(size_t)1023;
        const size_t stage_bytes = (size_t)(SN_TILE_H + 2) * SN_TILE_W * row_bytes;
        // carries [epilogue warp][4][16] + bias [n_co] + statistics [4][2][n_co] floats
        const size_t extra = (size_t)(4 * pl.n_tile * 4 + pl.n_tile + (bn_sums != nullptr ? 4 * 2 * pl.n_tile : 0)) * sizeof(float) + 1024;
        static const int stages_sn = [] { const char* e = getenv("UAPS_CONV_SN_STAGES"); return e ? atoi(e) : 6; }();
        int stages = stages_sn >= 2 && stages_sn <= MAX_STAGES ? stages_sn : 6;
        for (;;) {
            while (stages > 2 && w_region + stages * stage_bytes + extra + 2048 > (size_t)(227 * 1024) / per_sm) --stages;
            if (w_region + stages * stage_bytes + extra + 2048 <= (size_t)(227 * 1024) / per_sm || per_sm == 1) break;
            --per_sm;                                      // two stages do not fit this many CTAs: fewer CTAs, more stages
            stages = stages_sn >= 2 && stages_sn <= MAX_STAGES ? stages_sn : 6;
        }
        a.stages = stages;
        const size_t smem = w_region + stages * stage_bytes + extra;
        if (smem > 227 * 1024) return UAPS_ERANGE;
        cudaError_t e;
        int occ = 0;
        // (cudaOccupancyMaxActiveBlocksPerMultiprocessor answered 1 for these kernels on B200 where 3 CTAs run: the CTAs per SM
        // are derived from the kernel's register count instead)
#define UAPS_CONV_LAUNCH3(CKV, NGV)                                                                                          \
        e = cudaFuncSetAttribute(conv_sn_kernel<CKV, NGV>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);             \
        if (e != cudaSuccess) return (int)e;                                                                                     \
        {                                                                                                                        \
            static const int regs = [] {                                                                                         \
                cudaFuncAttributes fa{};                                                                                         \
                return cudaFuncGetAttributes(&fa, conv_sn_kernel<CKV, NGV>) == cudaSuccess ? fa.numRegs : 255;                   \
            }();                                                                                                                 \
            occ = 65536 / (((regs + 7) / 8 * 8) * SnCfg<NGV>::THREADS);                                                          \
        }                                                                                                                        \
        if (occ < 1) return UAPS_ERANGE;                                                                                         \
        if (per_sm > occ) per_sm = occ;                    /* registers: the TMEM columns of more CTAs would never be freed */   \
        if (getenv("UAPS_CONV_DEBUG") != nullptr)                                                                                \
            fprintf(stderr, "conv_sn<%d,%d>: per_sm %d (regs allow %d) stages %d smem %zu units %d\n", CKV, NGV, per_sm, occ,     \
                    stages, smem, a.num_tiles);                                                                                  \
        gridx = (long long)device_info().sm_count * per_sm;                                                                      \
        if (gridx > a.num_tiles) gridx = a.num_tiles;                                                                            \
        UAPS_LAUNCH((conv_sn_kernel<CKV, NGV>), dim3((unsigned)gridx), dim3(SnCfg<NGV>::THREADS), smem, stream, m0, m1, a);
#define UAPS_CONV_LAUNCH3_NG(CKV)                                                                       \
        if (ng == 1) { UAPS_CONV_LAUNCH3(CKV, 1) } else if (ng == 2) { UAPS_CONV_LAUNCH3(CKV, 2) }         \
        else if (ng == 3) { UAPS_CONV_LAUNCH3(CKV, 3) } else { UAPS_CONV_LAUNCH3(CKV, 4) }
        long long gridx = 0;
        if (pl.ck == 64) { UAPS_CONV_LAUNCH3_NG(64) } else if (pl.ck == 32) { UAPS_CONV_LAUNCH3_NG(32) } else { UAPS_CONV_LAUNCH3_NG(16) }
#undef UAPS_CONV_LAUNCH3_NG
#undef UAPS_CONV_LAUNCH3
        UAPS_LAUNCH_CHECK();
        return UAPS_OK;
    }

    static const bool use_v1 = getenv("UAPS_CONV_V1") != nullptr;       // A/B knobs for profiling, not part of the ABI
    static const bool no_xhalo = getenv("UAPS_CONV_NO_XHALO") != nullptr;
    const int wbytes_all = pl.iters * b_bytes;
    a.resident = (!use_v1 && pl.n_tiles == 1 && wbytes_all <= W_RESIDENT_MAX) ? 1 : 0;
    a.xhalo = (a.resident && ks == 3 && !no_xhalo) ? 1 : 0;
    const int box_w = a.xhalo ? TILE_W + 2 : TILE_W;
    CUtensorMap m0, m1;
    rc = encode_map(&m0, x1, B, H, W, c1_stride, pl.ck, TILE_H + ks - 1, box_w);
    if (rc != UAPS_OK) return rc;
    rc = encode_map(&m1, cin2 > 0 ? x2 : x1, B, H, W, cin2 > 0 ? c2_stride : c1_stride, pl.ck, TILE_H + ks - 1, box_w);
    if (rc != UAPS_OK) return rc;

    cudaError_t e;
    if (use_v1) {
        const int stage_bytes = (a_bytes + b_bytes + 1023) & ~1023;
        int stages = pl.iters < 4 ? pl.iters : 4;
        while (stages > 1 && (size_t)stages * stage_bytes > 200 * 1024) --stages;
        a.stages = stages;
        const size_t smem = (size_t)stages * stage_bytes + 1024;
        dim3 grid((unsigned)(a.tiles_x * a.tiles_y * B), (unsigned)pl.n_tiles, 1);
#define UAPS_CONV_LAUNCH(CKV)                                                                                   \
        e = cudaFuncSetAttribute(conv_igemm_kernel<CKV>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);   \
        if (e != cudaSuccess) return (int)e;                                                                        \
        UAPS_LAUNCH(conv_igemm_kernel<CKV>, grid, dim3(THREADS), smem, stream, m0, m1, a);
        if (pl.ck == 64) { UAPS_CONV_LAUNCH(64) } else if (pl.ck == 32) { UAPS_CONV_LAUNCH(32) } else { UAPS_CONV_LAUNCH(16) }
#undef UAPS_CONV_LAUNCH
    } else {
        // persistent kernel: weights resident when they fit; as many stages as a budget of ~100 KB per CTA gives
        const int w_region = a.resident ? ((wbytes_all + 1023) & ~1023) : 0;
        const int a_bytes2 = (TILE_H + ks - 1) * box_w * row_bytes;
        const int stage_bytes = (a_bytes2 + (a.resident ? 0 : b_bytes) + 1023) & ~1023;
        static const int stages_env = [] { const char* e = getenv("UAPS_CONV_STAGES"); return e ? atoi(e) : 4; }();
        int stages = stages_env >= 2 && stages_env <= MAX_STAGES ? stages_env : 4;
        while (stages > 2 && (size_t)w_region + (size_t)stages * stage_bytes > 110 * 1024) --stages;
        if ((size_t)w_region + (size_t)stages * stage_bytes > 220 * 1024) stages = 2;
        while (stages > 1 && (size_t)w_region + (size_t)stages * stage_bytes > 220 * 1024) --stages;
        a.stages = stages;
        const size_t stat_bytes = bn_sums != nullptr ? (size_t)4 * 2 * pl.n_tile * sizeof(float) : 0;   // BN-statistics scratch
        const size_t smem = (size_t)w_region + (size_t)stages * stage_bytes + stat_bytes + 1024;
        int tmem_cols = 32;
        while (tmem_cols < 2 * pl.n_tile) tmem_cols <<= 1;
        int per_sm = (int)((227 * 1024) / (smem + 2048));
        if (per_sm > 512 / tmem_cols) per_sm = 512 / tmem_cols;
        // measured on B200 (16-channel layers, B=64): 4 CTAs/SM 88 us, 6 -> 80 us, 8 -> 99 us
        static const int cap_env = [] { const char* e = getenv("UAPS_CONV_CTAS_PER_SM"); return e ? atoi(e) : 6; }();
    if (per_sm > cap_env) per_sm = cap_env;
        if (per_sm < 1) per_sm = 1;
        long long gridx = (long long)device_info().sm_count * per_sm;
        if (gridx > a.num_tiles) gridx = a.num_tiles;
        if (bn_sums != nullptr && pl.n_tiles > 1) {          // every CTA must see ONE output-channel block (its statistics columns)
            gridx = gridx / pl.n_tiles * pl.n_tiles;
            if (gridx < pl.n_tiles) gridx = pl.n_tiles;
        }
        if (getenv("UAPS_CONV_DEBUG") != nullptr)
            fprintf(stderr, "conv_persistent<%d>: per_sm %d stages %d smem %zu grid %lld num_tiles %d\n", pl.ck, per_sm, stages,
                    smem, gridx, a.num_tiles);
#define UAPS_CONV_LAUNCH2(CKV)                                                                                           \
        e = cudaFuncSetAttribute(conv_igemm_persistent_kernel<CKV>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);   \
        if (e != cudaSuccess) return (int)e;                                                                                   \
        UAPS_LAUNCH(conv_igemm_persistent_kernel<CKV>, dim3((unsigned)gridx), dim3(THREADS2), smem, stream, m0, m1, a);
        if (pl.ck == 64) { UAPS_CONV_LAUNCH2(64) } else if (pl.ck == 32) { UAPS_CONV_LAUNCH2(32) } else { UAPS_CONV_LAUNCH2(16) }
#undef UAPS_CONV_LAUNCH2
    }
    UAPS_LAUNCH_CHECK();
    return UAPS_OK;
}
}  // namespace
