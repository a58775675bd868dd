// Validation head: the per-batch quantities of the reference's validation pass (UAPS_train.py:377-385) from the main
// decoder's logits in one read -- the confusion matrix behind pixel accuracy / mIoU / mDice (utilities/metrics.py) and
// the cross-entropy sum of CrossEntropyLoss() (:75, ignore_index -100) -- then one fold that appends the batch as a row
// of a caller-owned epoch table.  See include/uaps_b200.h for the contract and DESIGN.md f6 for the numbers.
// uaps_val_scalars copies a few device scalars (a training iteration's losses, DESIGN.md f9) into the row of a second
// table that the fold has just written, so the two tables stay row-aligned without the host.
//
// Grid as the ensemble head (ensemble_head.cu): blockIdx.y = image, blockIdx.x = a fixed span of that image's pixels.
// The span is counted in pixels, so the number of blocks depends on (B, HW) only and uaps_val_fold can recompute it.
// Every block writes its own partial record (no atomics on global memory, nothing to zero between calls); the fold adds
// them in a fixed order, so a row is bitwise reproducible and both launches can be captured into a CUDA graph.
#include "argmax_exact.cuh"

namespace uaps {
namespace val {

constexpr int THREADS = 128;
constexpr int WARPS = THREADS / kWarp;
constexpr int TARGET_BLOCKS = 2048;    // a thread takes 2 or 4 pixel groups per chunk only while the grid keeps this many blocks
constexpr int FOLD_THREADS = 512;
constexpr long long IGNORE = -100;     // torch's default ignore_index

// pixels of one image a block covers: 4 pixels per thread and iteration whatever the vector width
inline long long span_pixels(int B, int64_t HW) {
    const long long total = (long long)B * HW;
    const long long per = 4LL * THREADS * TARGET_BLOCKS;
    return 4LL * THREADS * (total >= 4 * per ? 4 : (total >= 2 * per ? 2 : 1));
}
inline unsigned chunks_per_image(int B, int64_t HW) { return (unsigned)ceil_div<long long>(HW, span_pixels(B, HW)); }

// workspace: double ce[nblk] | uint32 words[C*C + 2][nblk] (word-major, so the fold reads each word coalesced):
// words 0..C*C-1 the confusion counts (label * C + prediction), C*C the non-ignored pixels, C*C+1 the bad labels
inline size_t workspace_bytes(int C, int B, int64_t HW) {
    const size_t nblk = (size_t)B * chunks_per_image(B, HW);
    return nblk * sizeof(double) + (size_t)(C * C + 2) * nblk * sizeof(uint32_t);
}

struct CountArgs {
    const float* z;            // [B, C, HW]
    const long long* labels;   // [B, HW]
    double* ce;
    uint32_t* words;
    long long HW;
    unsigned groups_per_image; // HW / VEC
    unsigned span_groups;      // pixel groups per chunk
    unsigned nblk;
};

template <int VEC>
__device__ __forceinline__ void load_labels(const long long* p, long long (&l)[VEC]) {
    if constexpr (VEC == 1) {
        l[0] = __ldg(p);
    } else {
#pragma unroll
        for (int j = 0; j < VEC; j += 2) {
            const longlong2 v = __ldg(reinterpret_cast<const longlong2*>(p + j));
            l[j] = v.x; l[j + 1] = v.y;
        }
    }
}

template <int C, int VEC>
__global__ void __launch_bounds__(THREADS) val_counts_kernel(const __grid_constant__ CountArgs a) {
    __shared__ unsigned s_conf[WARPS][C * C];      // one histogram per warp: fewer shared-atomic collisions
    __shared__ double s_ce[WARPS];
    __shared__ unsigned s_n[WARPS][2];
    grid_dep_launch();
    for (int i = threadIdx.x; i < WARPS * C * C; i += THREADS) (&s_conf[0][0])[i] = 0u;
    __syncthreads();
    grid_dep_wait();                               // the logits are the previous kernel's output (out_conv)
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const unsigned b = blockIdx.y;
    const unsigned g_end = min(blockIdx.x * a.span_groups + a.span_groups, a.groups_per_image);
    double ce = 0.0;
    unsigned valid = 0, bad = 0;
    for (unsigned g = blockIdx.x * a.span_groups + threadIdx.x; g < g_end; g += THREADS) {
        const size_t hw = (size_t)g * VEC;
        const size_t base = (size_t)b * C * a.HW + hw;
        float zv[C][VEC];
#pragma unroll
        for (int c = 0; c < C; ++c) load_vec<VEC>(a.z + base + (size_t)c * a.HW, zv[c]);
        long long lab[VEC];
        load_labels<VEC>(a.labels + (size_t)b * a.HW + hw, lab);
#pragma unroll
        for (int j = 0; j < VEC; ++j) {
            float z[C];
#pragma unroll
            for (int c = 0; c < C; ++c) z[c] = zv[c][j];
            const int pred = argmax_softmax<C>(z);
            const long long l = lab[j];
            if (l >= 0 && l < C) {
                // -log_softmax(z)[l] = log(sum exp(z - m)) - (z[l] - m), fp32 as torch's log_softmax; the max and the
                // exponentials are those of argmax_softmax (the compiler shares them)
                float m = z[0];
#pragma unroll
                for (int c = 1; c < C; ++c) m = fmaxf(m, z[c]);
                float s = 0.f, zl = z[0];
#pragma unroll
                for (int c = 0; c < C; ++c) {
                    s = __fadd_rn(s, expf(__fsub_rn(z[c], m)));
                    if (c == (int)l) zl = z[c];
                }
                ce += (double)__fsub_rn(logf(s), __fsub_rn(zl, m));
                ++valid;
                atomicAdd(&s_conf[warp][(int)l * C + pred], 1u);
            } else if (l != IGNORE) {
                ++bad;
            }
        }
    }
    // block partials in a fixed order: warp tree, then the warps in index order
    ce = warp_sum(ce);
    valid = __reduce_add_sync(0xffffffffu, valid);
    bad = __reduce_add_sync(0xffffffffu, bad);
    if (lane == 0) { s_ce[warp] = ce; s_n[warp][0] = valid; s_n[warp][1] = bad; }
    __syncthreads();
    const unsigned blk = blockIdx.y * gridDim.x + blockIdx.x;
    for (int i = threadIdx.x; i < C * C; i += THREADS) {
        unsigned s = 0;
#pragma unroll
        for (int w = 0; w < WARPS; ++w) s += s_conf[w][i];
        a.words[(size_t)i * a.nblk + blk] = s;
    }
    if (threadIdx.x == 0) {
        double r = 0.0;
        unsigned v = 0, bb = 0;
#pragma unroll
        for (int w = 0; w < WARPS; ++w) { r += s_ce[w]; v += s_n[w][0]; bb += s_n[w][1]; }
        a.ce[blk] = r;
        a.words[(size_t)(C * C) * a.nblk + blk] = v;
        a.words[(size_t)(C * C + 1) * a.nblk + blk] = bb;
    }
}

// one block: the partials of all blocks in a fixed order -> row state[0] of the table, then state[0] += 1
__global__ void __launch_bounds__(FOLD_THREADS) val_fold_kernel(const double* __restrict__ ce, const uint32_t* __restrict__ words,
                                                                unsigned nblk, int C, double n_pixels, double* __restrict__ table,
                                                                unsigned max_batches, uint32_t* __restrict__ state) {
    __shared__ double s_ce[FOLD_THREADS / kWarp];
    __shared__ unsigned s_row;
    grid_dep_launch();
    grid_dep_wait();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int nw = C * C + 2, row_len = C * C + 3;
    double r = 0.0;
    for (unsigned i = threadIdx.x; i < nblk; i += FOLD_THREADS) r += __ldcg(ce + i);
    r = warp_sum(r);
    if (lane == 0) s_ce[warp] = r;
    if (threadIdx.x == 0) s_row = state[0];
    __syncthreads();
    const unsigned row = s_row;
    const bool ok = row < max_batches;
    double* out = table + (size_t)row * row_len;
    for (int w = warp; w < nw; w += FOLD_THREADS / kWarp) {   // integer sums: any order gives the same result
        const uint32_t* src = words + (size_t)w * nblk;
        unsigned s = 0;
#pragma unroll 8
        for (unsigned i = lane; i < nblk; i += kWarp) s += __ldcg(src + i);
        s = __reduce_add_sync(0xffffffffu, s);
        if (lane == 0) {
            if (w == nw - 1) state[2] += s;                              // bad labels: latched for the whole table
            else if (ok) out[w < C * C ? w : C * C + 1] = (double)s;     // counts | non-ignored pixels
        }
    }
    if (threadIdx.x == 0) {
        if (ok) {
            double t = 0.0;
#pragma unroll
            for (int w = 0; w < FOLD_THREADS / kWarp; ++w) t += s_ce[w];
            out[C * C] = t;
            out[C * C + 2] = n_pixels;
            state[0] = row + 1;
        } else {
            state[1] = 1u;                                               // overflow: the batch is not recorded
        }
    }
}

struct ScalarSrc { const float* p[UAPS_VAL_SCALARS_MAX]; };

// one warp: scalar i -> table[state[0] - 1][i], the row the preceding fold on the same state wrote
__global__ void __launch_bounds__(kWarp) val_scalars_kernel(const __grid_constant__ ScalarSrc src, int n,
                                                            double* __restrict__ table, unsigned max_rows,
                                                            const uint32_t* __restrict__ state) {
    grid_dep_launch();
    grid_dep_wait();
    const unsigned row = state[0];
    if (state[1] != 0u || row == 0u || row > max_rows || (int)threadIdx.x >= n) return;   // overflow: nothing recorded
    table[(size_t)(row - 1) * n + threadIdx.x] = (double)*src.p[threadIdx.x];
}

template <int C, int VEC>
int launch_counts(CountArgs a, int B, cudaStream_t st) {
    a.groups_per_image = (unsigned)(a.HW / VEC);
    a.span_groups = (unsigned)(span_pixels(B, a.HW) / VEC);
    const unsigned chunks = chunks_per_image(B, a.HW);
    a.nblk = (unsigned)B * chunks;
    UAPS_LAUNCH((val_counts_kernel<C, VEC>), dim3(chunks, B), dim3(THREADS), 0, st, a);
    return UAPS_OK;
}

template <int C>
int launch_c(int vec, const CountArgs& a, int B, cudaStream_t st) {
    if (vec == 4) return launch_counts<C, 4>(a, B, st);
    if (vec == 2) return launch_counts<C, 2>(a, B, st);
    return launch_counts<C, 1>(a, B, st);
}

int check_sizes(int B, int C, int64_t HW) {
    if (B <= 0 || HW <= 0) return UAPS_EINVAL;
    if (C < 2 || C > UAPS_CMAX) return UAPS_ERANGE;
    if ((double)B * (double)HW >= 2147483648.0 || B > 65535) return UAPS_ERANGE;
    return UAPS_OK;
}

}  // namespace val
}  // namespace uaps

using namespace uaps;

UAPS_API size_t uaps_val_workspace_bytes(int C, int B, int64_t HW) {
    if (val::check_sizes(B, C, HW) != UAPS_OK) return 0;
    return val::workspace_bytes(C, B, HW);
}

UAPS_API int uaps_val_counts(const float* logits, const int64_t* labels, int B, int C, int64_t HW, void* workspace,
                             size_t workspace_bytes, cudaStream_t stream) {
    if (logits == nullptr || labels == nullptr || workspace == nullptr) return UAPS_EINVAL;
    const int rc = val::check_sizes(B, C, HW);
    if (rc != UAPS_OK) return rc;
    if (!aligned_to(logits, 4) || !aligned_to(labels, 8) || !aligned_to(workspace, 8)) return UAPS_EALIGN;
    if (workspace_bytes < val::workspace_bytes(C, B, HW)) return UAPS_EINVAL;
    // widest vector width the plane length and both pointers allow (as the ensemble head picks it)
    int vec = (HW % 4 == 0) ? 4 : (HW % 2 == 0 ? 2 : 1);
    while (vec > 1 && !aligned_to(logits, 4 * (size_t)vec)) vec >>= 1;
    if (vec > 1 && !aligned_to(labels, 16)) vec = 1;
    const size_t nblk = (size_t)B * val::chunks_per_image(B, HW);
    val::CountArgs a{};
    a.z = logits;
    a.labels = reinterpret_cast<const long long*>(labels);
    a.ce = reinterpret_cast<double*>(workspace);
    a.words = reinterpret_cast<uint32_t*>(a.ce + nblk);
    a.HW = HW;
    switch (C) {
        case 2: return val::launch_c<2>(vec, a, B, stream);
        case 3: return val::launch_c<3>(vec, a, B, stream);
        case 4: return val::launch_c<4>(vec, a, B, stream);
        case 5: return val::launch_c<5>(vec, a, B, stream);
        case 6: return val::launch_c<6>(vec, a, B, stream);
        case 7: return val::launch_c<7>(vec, a, B, stream);
        case 8: return val::launch_c<8>(vec, a, B, stream);
    }
    return UAPS_ERANGE;
}

UAPS_API int uaps_val_fold(const void* workspace, size_t workspace_bytes, int B, int C, int64_t HW, double* table,
                           int max_batches, uint32_t* state, cudaStream_t stream) {
    if (workspace == nullptr || table == nullptr || state == nullptr || max_batches < 0) return UAPS_EINVAL;
    const int rc = val::check_sizes(B, C, HW);
    if (rc != UAPS_OK) return rc;
    if (!aligned_to(workspace, 8) || !aligned_to(table, 8) || !aligned_to(state, 4)) return UAPS_EALIGN;
    if (workspace_bytes < val::workspace_bytes(C, B, HW)) return UAPS_EINVAL;
    const unsigned nblk = (unsigned)B * val::chunks_per_image(B, HW);
    const double* ce = reinterpret_cast<const double*>(workspace);
    const uint32_t* words = reinterpret_cast<const uint32_t*>(ce + nblk);
    UAPS_LAUNCH(val::val_fold_kernel, dim3(1), dim3(val::FOLD_THREADS), 0, stream, ce, words, nblk, C,
                (double)B * (double)HW, table, (unsigned)max_batches, state);
    return UAPS_OK;
}

UAPS_API int uaps_val_scalars(const float* const* src, int n, double* table, int max_rows, const uint32_t* state,
                              cudaStream_t stream) {
    if (src == nullptr || table == nullptr || state == nullptr || max_rows < 0) return UAPS_EINVAL;
    if (n < 1 || n > UAPS_VAL_SCALARS_MAX) return UAPS_ERANGE;
    if (!aligned_to(table, 8) || !aligned_to(state, 4)) return UAPS_EALIGN;
    val::ScalarSrc s{};
    for (int i = 0; i < n; ++i) {
        if (src[i] == nullptr) return UAPS_EINVAL;
        if (!aligned_to(src[i], 4)) return UAPS_EALIGN;
        s.p[i] = src[i];
    }
    UAPS_LAUNCH(val::val_scalars_kernel, dim3(1), dim3(kWarp), 0, stream, s, n, table, (unsigned)max_rows, state);
    return UAPS_OK;
}
