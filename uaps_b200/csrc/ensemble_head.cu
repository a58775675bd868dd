// Ensemble inference head: K decoders' logits -> label map, per-pixel and per-image uncertainty, mean prediction.
// The test-time use of UAPS's auxiliary decoders (UAPS-Testing.ipynb cell 11): the same per-pixel softmax / mean
// prediction / KL arithmetic as pass 1 of the fused loss (fused_loss_impl.cuh, reused, not copied), without the loss
// sums.  See include/uaps_b200.h for the contract and DESIGN.md f5 for the numbers.
//
// Grid: blockIdx.y = image, blockIdx.x = a fixed span of that image's pixels (a chunk), so each block owns one
// image's pixels only and the per-image uncertainty sum is a fixed-order fold of per-chunk fp64 partials -- bitwise
// reproducible, no atomics, nothing to zero between calls (graph-capturable).
#include "fused_loss_impl.cuh"

namespace uaps {
namespace ens {
using namespace loss;

constexpr int THREADS = 128;
constexpr int TARGET_BLOCKS = 2048;   // a thread takes 2 or 4 pixel groups per chunk only while the grid keeps this many blocks (~14 per SM)

// CTAs per SM the register allocator is asked to fit: the loss's estimate (min_ctas) holds the logits and its running
// sums; the head instead keeps every decoder's p and log p of a pixel live until its mean prediction is known
__host__ __device__ constexpr int head_min_ctas(int K, int C, int VEC) {
    const int need = K * C * VEC + 2 * K * C + 2 * C + 64;
    return need <= 124 ? 4 : (need <= 168 ? 3 : 2);
}

struct EnsArgs {
    const float* z[KMAX];        // K logits [B, C, HW] fp32
    uint8_t* labels;             // [B, HW]
    float* unc;                  // nullable [B, HW]
    float* q;                    // nullable [B, C, HW]
    double* partials;            // nullable [B][chunks]: per-chunk sums of the uncertainty map
    long long HW;
    unsigned groups_per_image;   // HW / VEC
    unsigned iters;              // pixel groups per thread per chunk
};

template <int VEC>
__device__ __forceinline__ void store_labels(uint8_t* p, const int (&y)[VEC]) {
    if constexpr (VEC == 4) {
        *reinterpret_cast<uint32_t*>(p) = (uint32_t)y[0] | ((uint32_t)y[1] << 8) | ((uint32_t)y[2] << 16) | ((uint32_t)y[3] << 24);
    } else if constexpr (VEC == 2) {
        *reinterpret_cast<uint16_t*>(p) = (uint16_t)((uint32_t)y[0] | ((uint32_t)y[1] << 8));
    } else {
        *p = (uint8_t)y[0];
    }
}

// PF: the next pixel group's K*C loads are issued before this one is computed (as in loss pass 1)
template <int K, int C, int VEC, bool PF>
__global__ void __launch_bounds__(THREADS, head_min_ctas(K, C, PF ? 2 * VEC : VEC))
ensemble_head_kernel(const __grid_constant__ EnsArgs a) {
    __shared__ double s_red[THREADS / kWarp];
    pdl_wait();                       // the logits may be the previous kernel's output (out_conv epilogue)
    pdl_trigger();
    const unsigned b = blockIdx.y;
    const unsigned gbase = b * a.groups_per_image;
    const unsigned span = a.iters * THREADS;
    const unsigned g_end = min(blockIdx.x * span + span, a.groups_per_image);
    unsigned g = blockIdx.x * span + threadIdx.x;
    double img = 0.0;
    float zn[PF ? K : 1][PF ? C : 1][PF ? VEC : 1];
    if constexpr (PF) { if (g < g_end) load_group<K, C, VEC>(a, gbase + g, zn); }
    for (; g < g_end; g += THREADS) {
        float zv[K][C][VEC];
        if constexpr (PF) {
#pragma unroll
            for (int k = 0; k < K; ++k)
#pragma unroll
                for (int c = 0; c < C; ++c)
#pragma unroll
                    for (int j = 0; j < VEC; ++j) zv[k][c][j] = zn[k][c][j];
            if (g + THREADS < g_end) load_group<K, C, VEC>(a, gbase + g + THREADS, zn);
        } else {
            load_group<K, C, VEC>(a, gbase + g, zv);
        }
        const size_t hw = (size_t)g * VEC;
        const size_t base = (size_t)b * C * a.HW + hw;
        int yv[VEC];
        float uv[VEC];
        float qv[C][VEC];
#pragma unroll
        for (int j = 0; j < VEC; ++j) {
            float z[K][C];
#pragma unroll
            for (int k = 0; k < K; ++k)
#pragma unroll
                for (int c = 0; c < C; ++c) z[k][c] = zv[k][c][j];
            PixelState<K, C> st;
            pixel_mean_forward<K, C>(z, a, base + j, st);
            float vs = st.V[0];
#pragma unroll
            for (int k = 1; k < K; ++k) vs += st.V[k];
            yv[j] = st.y;
            uv[j] = mean_of_sum<K>(vs);                                   // (1/K) sum_k V_k (UAPS_train.py:241)
            img += (double)uv[j];
#pragma unroll
            for (int c = 0; c < C; ++c) qv[c][j] = st.q[c];
        }
        const size_t pix = (size_t)b * a.HW + hw;
        store_labels<VEC>(a.labels + pix, yv);
        if (a.unc != nullptr) store_vec<VEC>(a.unc + pix, uv);
        if (a.q != nullptr) {
#pragma unroll
            for (int c = 0; c < C; ++c) store_vec<VEC>(a.q + base + (size_t)c * a.HW, qv[c]);
        }
    }
    if (a.partials != nullptr) {      // block sum in a fixed order: warp tree, then the warps in index order
        const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
        img = warp_sum(img);
        if (lane == 0) s_red[warp] = img;
        __syncthreads();
        if (threadIdx.x == 0) {
            double r = 0.0;
#pragma unroll
            for (int w = 0; w < THREADS / kWarp; ++w) r += s_red[w];
            a.partials[(size_t)b * gridDim.x + blockIdx.x] = r;
        }
    }
}

// one warp per image: its chunk partials in a fixed order (lane-strided, then a shuffle tree), mean over HW
__global__ void __launch_bounds__(256) ensemble_image_fold_kernel(const double* __restrict__ partials, int B, unsigned chunks,
                                                                  double inv_hw, float* __restrict__ out) {
    pdl_wait();
    const int lane = threadIdx.x & 31;
    const int b = blockIdx.x * (256 / kWarp) + (threadIdx.x >> 5);
    if (b >= B) return;
    double r = 0.0;
    for (unsigned i = lane; i < chunks; i += kWarp) r += __ldcg(partials + (size_t)b * chunks + i);
    r = warp_sum(r);
    if (lane == 0) out[b] = (float)(r * inv_hw);
}

template <int K, int C, int VEC, bool PF>
int launch_vec(EnsArgs a, int B, float* image_unc, unsigned* chunks_out, bool dry, cudaStream_t st) {
    a.groups_per_image = (unsigned)(a.HW / VEC);
    const long long total = (long long)B * a.groups_per_image;
    a.iters = total >= 4LL * THREADS * TARGET_BLOCKS ? 4u : (total >= 2LL * THREADS * TARGET_BLOCKS ? 2u : 1u);
    const unsigned chunks = (unsigned)ceil_div<long long>(a.groups_per_image, (long long)a.iters * THREADS);
    *chunks_out = chunks;
    if (dry) return UAPS_OK;
    cudaError_t e = launch_pdl(ensemble_head_kernel<K, C, VEC, PF>, dim3(chunks, B), dim3(THREADS), st, pdl_enabled(), a);
    if (e != cudaSuccess) return (int)e;
    if (image_unc != nullptr) {
        e = launch_pdl(ensemble_image_fold_kernel, dim3(ceil_div(B, 256 / kWarp)), dim3(256), st, pdl_enabled(),
                       (const double*)a.partials, B, chunks, 1.0 / (double)a.HW, image_unc);
        if (e != cudaSuccess) return (int)e;
    }
    UAPS_LAUNCH_CHECK();
    return UAPS_OK;
}

template <int K, int C>
int launch_kc(int vec, const EnsArgs& a, int B, float* image_unc, unsigned* chunks, bool dry, cudaStream_t st) {
    if constexpr (has_vec4(K, C)) { if (vec == 4) return launch_vec<K, C, 4, true>(a, B, image_unc, chunks, dry, st); }
    if constexpr (has_vec2(K, C)) { if (vec >= 2) return launch_vec<K, C, 2, true>(a, B, image_unc, chunks, dry, st); }
    return launch_vec<K, C, 1, false>(a, B, image_unc, chunks, dry, st);
}

template <int K>
int launch_for_k(int C, int vec, const EnsArgs& a, int B, float* image_unc, unsigned* chunks, bool dry, cudaStream_t st) {
    switch (C) {
        case 2: return launch_kc<K, 2>(vec, a, B, image_unc, chunks, dry, st);
        case 3: return launch_kc<K, 3>(vec, a, B, image_unc, chunks, dry, st);
        case 4: return launch_kc<K, 4>(vec, a, B, image_unc, chunks, dry, st);
        case 5: return launch_kc<K, 5>(vec, a, B, image_unc, chunks, dry, st);
        case 6: return launch_kc<K, 6>(vec, a, B, image_unc, chunks, dry, st);
        case 7: return launch_kc<K, 7>(vec, a, B, image_unc, chunks, dry, st);
        case 8: return launch_kc<K, 8>(vec, a, B, image_unc, chunks, dry, st);
    }
    return UAPS_ERANGE;
}

int dispatch(int K, int C, int vec, const EnsArgs& a, int B, float* image_unc, unsigned* chunks, bool dry, cudaStream_t st) {
    switch (K) {
        case 1: return launch_for_k<1>(C, vec, a, B, image_unc, chunks, dry, st);
        case 2: return launch_for_k<2>(C, vec, a, B, image_unc, chunks, dry, st);
        case 3: return launch_for_k<3>(C, vec, a, B, image_unc, chunks, dry, st);
        case 4: return launch_for_k<4>(C, vec, a, B, image_unc, chunks, dry, st);
        case 5: return launch_for_k<5>(C, vec, a, B, image_unc, chunks, dry, st);
        case 6: return launch_for_k<6>(C, vec, a, B, image_unc, chunks, dry, st);
    }
    return UAPS_ERANGE;
}

}  // namespace ens
}  // namespace uaps

using namespace uaps;

UAPS_API size_t uaps_ensemble_workspace_bytes(int K, int C, int B, int64_t HW) {
    if (K < 1 || K > UAPS_KMAX || C < 2 || C > UAPS_CMAX || B <= 0 || HW <= 0) return 0;
    // the most chunks any launch makes: one pixel group of one pixel per thread
    return (size_t)B * (size_t)ceil_div<int64_t>(HW, ens::THREADS) * sizeof(double);
}

UAPS_API int uaps_ensemble_head(const float* const* z, int K, int B, int C, int64_t HW, uint8_t* labels, float* uncertainty,
                                float* image_uncertainty, float* mean_prob, void* workspace, size_t workspace_bytes,
                                cudaStream_t stream) {
    if (z == nullptr || labels == nullptr || B <= 0 || HW <= 0) return UAPS_EINVAL;
    if (K < 1 || K > UAPS_KMAX || C < 2 || C > UAPS_CMAX) return UAPS_ERANGE;
    if ((double)B * (double)HW >= 2147483648.0 || B > 65535) return UAPS_ERANGE;
    ens::EnsArgs a{};
    // widest vector width the plane length and every pointer allow (as the loss picks it)
    int vec = (HW % 4 == 0) ? 4 : (HW % 2 == 0 ? 2 : 1);
    auto narrow = [&vec](const void* p, int bytes_per_pixel) {
        while (vec > 1 && !aligned_to(p, (size_t)bytes_per_pixel * vec)) vec >>= 1;
    };
    for (int k = 0; k < K; ++k) {
        if (z[k] == nullptr) return UAPS_EINVAL;
        if (!aligned_to(z[k], 4)) return UAPS_EALIGN;
        a.z[k] = z[k];
        narrow(z[k], 4);
    }
    if ((uncertainty != nullptr && !aligned_to(uncertainty, 4)) || (mean_prob != nullptr && !aligned_to(mean_prob, 4)) ||
        (image_uncertainty != nullptr && !aligned_to(image_uncertainty, 4)))
        return UAPS_EALIGN;
    narrow(labels, 1);
    if (uncertainty != nullptr) narrow(uncertainty, 4);
    if (mean_prob != nullptr) narrow(mean_prob, 4);
    a.labels = labels; a.unc = uncertainty; a.q = mean_prob; a.HW = HW;
    if (image_uncertainty != nullptr) {
        if (workspace == nullptr) return UAPS_EINVAL;
        if (!aligned_to(workspace, 8)) return UAPS_EALIGN;
        unsigned chunks = 0;
        const int rc = ens::dispatch(K, C, vec, a, B, nullptr, &chunks, true, stream);    // dry run: the grid's chunk count
        if (rc != UAPS_OK) return rc;
        if (workspace_bytes < (size_t)B * chunks * sizeof(double)) return UAPS_EINVAL;
        a.partials = reinterpret_cast<double*>(workspace);
    }
    unsigned chunks = 0;
    return ens::dispatch(K, C, vec, a, B, image_uncertainty, &chunks, false, stream);
}
