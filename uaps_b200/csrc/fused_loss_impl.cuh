// Fused pseudo-label + KL-uncertainty + uncertainty-weighted CE/Dice loss, forward (pass 1),
// scalar finalize, and backward (pass 2).  Replaces UAPS_train.py:186-189, 223-282 (+ :194-218 in
// supervised mode) and their autograd graph.  See include/uaps_b200.h for the ABI contract and
// DESIGN.md §3 for the math.
//
// Data layout: K logits tensors, each contiguous NCHW fp32.  A thread owns VEC consecutive pixels
// of one image and issues K*C independent 128-bit loads (one per class plane) before any math,
// so a warp has K*C*512 B in flight per iteration; all per-pixel state lives in registers.
//
// Bit-exactness of the pseudo-label: the chain that decides argmax reproduces the op order and
// roundings of torch's CUDA kernels -- max, x-max, expf, sequential sum, IEEE divide
// (cunn_SpatialSoftMaxForward), then separately rounded w*p multiplies and left-associated adds
// (one ATen kernel each in the reference, so no FMA contraction), then first-maximum argmax.
#pragma once
#include <cstdlib>
#include "common.cuh"

namespace uaps {
namespace loss {

constexpr int KMAX = UAPS_KMAX;
constexpr int CMAX = UAPS_CMAX;
constexpr int LOSS_THREADS = 128;
constexpr int LOSS_MAX_BLOCKS = 640;            // >= 148 SMs x 4 CTAs; bounds the unrolled final fold
constexpr int WS_HEADER_BYTES = 256;          // ticket counter lives in the first 4 bytes

__host__ __device__ constexpr int sums_count(int K, int C) { return 3 * K + 2 * K * C + C; }
// CTAs (of 128 threads) per SM the register allocator is asked to fit: estimated live registers =
// the K*C*VEC logits + (pass 1) the running sums + ~64 of per-pixel state
__host__ __device__ constexpr int min_ctas(int K, int C, int VEC, bool pass1) {
#ifdef UAPS_P1_CTAS
    if (pass1) return UAPS_P1_CTAS;       // tuning experiments only
#endif
    const int need = K * C * VEC + (pass1 ? sums_count(K, C) : K * C) + 64;
    return need <= 124 ? 4 : (need <= 176 ? 3 : 2);
}
__host__ __device__ constexpr int scalars_count(int K, int C) { return UAPS_SC_BASE + 4 * K + 2 * K * C; }

// ---- programmatic dependent launch (PDL) ---------------------------------------------------------------------
// pass 1 -> fold/finalize -> pass 2 are launched with cudaLaunchAttributeProgrammaticStreamSerialization: a kernel's
// CTAs may become resident while its predecessor is still draining, and block in pdl_wait() until the predecessor
// has completed and flushed.  Everything a kernel reads that a predecessor may have written is read after pdl_wait();
// pass 2 issues its first logits loads before it (the logits were already consumed by pass 1 of the same loss, so they
// are older than any predecessor's output), which hides the fold/finalize kernel and two launch gaps behind them.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, cudaStream_t st, bool pdl, Args... args) {
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = 0; cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = pdl ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kern, KArgs(args)...);
}
inline bool pdl_enabled() {
    static const bool on = [] { const char* e = getenv("UAPS_LOSS_PDL"); return e == nullptr || atoi(e) != 0; }();
    return on;
}

struct LossArgs {
    const float* z[KMAX];
    float* out[KMAX];            // pass1: exp_var_out (nullable entries); pass2: dz
    float w[KMAX];
    const float* w_dev;          // nullable: device copy of the mix weights (UapsStepState.mix_w) that overrides w[]
    const int64_t* labels;       // supervised mode
    int64_t* pseudo;             // pass1 optional
    long long HW;
    unsigned groups_per_image;   // HW / VEC
    unsigned ngroups;            // B * groups_per_image
    int B;
    int write_ev;
};

// ---- per-pixel forward -------------------------------------------------------------------
// Logarithms are carried in a mode-dependent unit U: natural logs in EXACT mode (U = 1), log2 in the
// default mode (U = ln 2), so the MUFU results are used as they come and ln 2 is folded into the few
// consumers.
template <bool EXACT> struct LogUnit { static constexpr float U = EXACT ? 1.0f : 0.6931471805599453f; };

template <int K, int C>
struct PixelState {
    float p[K][C];   // softmax
    float l[K][C];   // log-softmax / U
    float q[C];      // mean prediction
    float lq[C];     // log q / U  (0 for q == 0 after kl_terms<GUARD>; see there)
    float V[K];      // KL(q || p_k) summed over classes
    float E[K];      // exp(-V)
    int y;           // pseudo-label / label
};

// EXACT: torch's op order and roundings (cunn_SpatialSoftMaxForward / LogSoftMax): max, x - max, expf,
// sequential sum, IEEE divide; log-softmax = (x - max) - logf(sum).
template <int C>
__device__ __forceinline__ void softmax_exact(const float (&z)[C], float (&p)[C], float (&l)[C]) {
    float m = z[0];
#pragma unroll
    for (int c = 1; c < C; ++c) m = fmaxf(m, z[c]);
    float e[C];
    float s = 0.f;
#pragma unroll
    for (int c = 0; c < C; ++c) {
        e[c] = expf(__fsub_rn(z[c], m));
        s = __fadd_rn(s, e[c]);
    }
    const float ls = logf(s);
#pragma unroll
    for (int c = 0; c < C; ++c) {
        p[c] = __fdiv_rn(e[c], s);
        l[c] = __fsub_rn(__fsub_rn(z[c], m), ls);
    }
}

// ---- default arithmetic: one MUFU per transcendental ------------------------------------------
// exp2/rcp/log2 approximations (<= 2 ulp) instead of the 10-20 instruction IEEE expansions.  Two
// things keep the results at the reference's accuracy:
//  * log p_kc is taken as lg2.approx(p_kc) itself, and log q_c as lg2.approx(q_c): the KL maps are
//    differences of the two, so the approximation's mantissa-dependent bias cancels (measured on
//    B200, tools/logbias.cu: mean-V error vs fp64 <= that of IEEE logf in every regime, while
//    t - lg2.approx(sum) is 10x worse when the decoders agree);
//  * the pseudo-label is still bit-exact: whenever the fast mix cannot separate the top two classes
//    by more than kTieMargin (>> the ~1.5e-6 worst-case distance between the fast and the torch-order
//    value) the argmax is re-decided from the logits with the exact torch-order chain.
__device__ __forceinline__ float ex2_approx(float x) { float y; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float lg2_approx(float x) { float y; asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float rcp_approx(float x) { float y; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
constexpr float kLog2e = 1.4426950408889634f;
constexpr float kTieMargin = 2e-5f;
constexpr float kLg2Floor = -120.0f;     // below this exp2 underflows (ftz): take log2 p from t - log2(sum) instead

template <int C, bool TRACK_MIN>
__device__ __forceinline__ float softmax_fast(const float (&z)[C], float (&p)[C], float (&l2)[C]) {
    float m = z[0];
#pragma unroll
    for (int c = 1; c < C; ++c) m = fmaxf(m, z[c]);
    const float nm = -m * kLog2e;          // a rounding error here scales every e_c alike and cancels in p
    float e[C];
    float s = 0.f, tmin = 0.f;
#pragma unroll
    for (int c = 0; c < C; ++c) {
        const float t = fmaf(z[c], kLog2e, nm);
        if constexpr (TRACK_MIN) tmin = fminf(tmin, t);
        e[c] = ex2_approx(t);
        s += e[c];
    }
    const float r = rcp_approx(s);
#pragma unroll
    for (int c = 0; c < C; ++c) {
        p[c] = e[c] * r;
        l2[c] = lg2_approx(p[c]);
    }
    return tmin;
}

// Rare fix-up (a class more than ~83 nats below its decoder's max): exp2 flushed p to 0, so take
// log2 p from (z - max) * log2(e) - log2(sum) like the reference's log-softmax does.
template <int C>
__device__ __forceinline__ void log2_softmax_underflow_fix(const float (&z)[C], float (&l2)[C]) {
    float m = z[0];
#pragma unroll
    for (int c = 1; c < C; ++c) m = fmaxf(m, z[c]);
    float t[C], s = 0.f;
#pragma unroll
    for (int c = 0; c < C; ++c) { t[c] = (z[c] - m) * kLog2e; s += ex2_approx(t[c]); }
    const float l2s = lg2_approx(s);
#pragma unroll
    for (int c = 0; c < C; ++c)
        if (t[c] < kLg2Floor) l2[c] = t[c] - l2s;      // lg2(p) is exact enough above the floor; below it p may have flushed
}

// torch's `acc / K` for the mean prediction (UAPS_train.py:223): ATen divides a CUDA tensor by a python scalar as a
// multiplication by the fp32-rounded reciprocal (div_true_kernel_cuda), so this is also what kl_terms computes
template <int K>
__device__ __forceinline__ float mean_of_sum(float acc) { return __fmul_rn(acc, 1.0f / K); }

// torch-order argmax of the Dirichlet mix (UAPS_train.py:251-255), every rounding reproduced
template <int K, int C>
__device__ __forceinline__ int argmax_exact(const float (&p)[K][C], const float (&w)[K]) {
    int y = 0;
    float best = 0.f;
#pragma unroll
    for (int c = 0; c < C; ++c) {
        float mix = __fmul_rn(w[0], p[0][c]);
#pragma unroll
        for (int k = 1; k < K; ++k) mix = __fadd_rn(mix, __fmul_rn(w[k], p[k][c]));
        if (c == 0) best = mix;
        else if (mix > best) { best = mix; y = c; }
    }
    return y;
}

// Near-tie slow path: re-reads the pixel's logits (L1/L2 hits) so the hot loop keeps nothing alive for it.
// MEAN: the argmax of the mean prediction q = (((p_0 + p_1) + p_2) + ...) / K (:223) instead of the mix, in the same
// torch order (the sum runs along the decoders, so only C partial sums stay live).  Args: LossArgs, or any argument
// block with the same z[] / HW fields (and w_dev / w unless MEAN).
template <int K, int C, bool MEAN = false, typename Args>
__device__ __noinline__ int argmax_exact_gmem(const Args& a, size_t pix_off) {
    if constexpr (MEAN) {
        float acc[C];
#pragma unroll
        for (int k = 0; k < K; ++k) {
            float z[C], p[C], l[C];
#pragma unroll
            for (int c = 0; c < C; ++c) z[c] = __ldg(a.z[k] + pix_off + (size_t)c * a.HW);
            softmax_exact<C>(z, p, l);
#pragma unroll
            for (int c = 0; c < C; ++c) acc[c] = k == 0 ? p[c] : __fadd_rn(acc[c], p[c]);
        }
        int y = 0;
        float best = mean_of_sum<K>(acc[0]);
#pragma unroll
        for (int c = 1; c < C; ++c) {
            const float q = mean_of_sum<K>(acc[c]);
            if (q > best) { best = q; y = c; }
        }
        return y;
    } else {
        float p[K][C], w[K];
#pragma unroll
        for (int k = 0; k < K; ++k) {
            float z[C], l[C];
#pragma unroll
            for (int c = 0; c < C; ++c) z[c] = __ldg(a.z[k] + pix_off + (size_t)c * a.HW);
            softmax_exact<C>(z, p[k], l);
            w[k] = a.w_dev != nullptr ? a.w_dev[k] : a.w[k];
        }
        return argmax_exact<K, C>(p, w);
    }
}

// mean prediction (UAPS_train.py:223) and KL maps (:226-236): V_k = sum_c xlogy(q,q) - q * l_kc, E_k = exp(-V_k).
// GUARD: apply xlogy's q == 0 -> 0 rule explicitly (the fast path leaves it to the NaN check of its caller), and give
// such a q a finite log, lq = 0.  lq is read again only by pass 2, in Gq_c, which enters dz only multiplied by p_kc
// <= K q_c: a -inf there made the pixel's dz NaN (0 * inf) where the limit is finite.  The default arithmetic's
// lg2.approx.ftz also flushes a subnormal q to -inf, so there the rule covers q < FLT_MIN (terms below 1e-36).
template <int K, int C, bool EXACT, bool GUARD>
__device__ __forceinline__ void kl_terms(PixelState<K, C>& st) {
    constexpr float U = LogUnit<EXACT>::U;
    float h = 0.f;
#pragma unroll
    for (int c = 0; c < C; ++c) {
        float acc = st.p[0][c];
#pragma unroll
        for (int k = 1; k < K; ++k) acc = __fadd_rn(acc, st.p[k][c]);
        const float q = acc * (1.0f / K);
        st.q[c] = q;
        if constexpr (GUARD) {
            const bool zero = EXACT ? q == 0.f : q < 1.17549435e-38f;
            st.lq[c] = zero ? 0.f : (EXACT ? logf(q) : lg2_approx(q));
            h += zero ? 0.f : q * st.lq[c];
        } else {
            st.lq[c] = EXACT ? logf(q) : lg2_approx(q);
            h = fmaf(q, st.lq[c], h);
        }
    }
#pragma unroll
    for (int k = 0; k < K; ++k) {
        float d = 0.f;
#pragma unroll
        for (int c = 0; c < C; ++c) d = fmaf(st.q[c], st.l[k][c], d);
        st.V[k] = (h - d) * U;
        st.E[k] = EXACT ? expf(-st.V[k]) : ex2_approx(-kLog2e * st.V[k]);
    }
}

template <int K, int C, bool SUP, bool EXACT>
__device__ __forceinline__ void pixel_forward(const float (&z)[K][C], const float (&w)[K], int label,
                                              const LossArgs& a, size_t pix_off, PixelState<K, C>& st) {
    if constexpr (EXACT) {
#pragma unroll
        for (int k = 0; k < K; ++k) softmax_exact<C>(z[k], st.p[k], st.l[k]);
        if constexpr (SUP) {
            st.y = label;
#pragma unroll
            for (int k = 0; k < K; ++k) { st.V[k] = 0.f; st.E[k] = 1.f; }
        } else {
            st.y = argmax_exact<K, C>(st.p, w);
            kl_terms<K, C, true, true>(st);
        }
    } else if constexpr (SUP) {
        float tmin = 0.f;
#pragma unroll
        for (int k = 0; k < K; ++k) tmin = fminf(tmin, softmax_fast<C, true>(z[k], st.p[k], st.l[k]));
        if (__builtin_expect(tmin < kLg2Floor, 0)) {
#pragma unroll
            for (int k = 0; k < K; ++k) log2_softmax_underflow_fix<C>(z[k], st.l[k]);
        }
        st.y = label;
#pragma unroll
        for (int k = 0; k < K; ++k) { st.V[k] = 0.f; st.E[k] = 1.f; }
    } else {
#pragma unroll
        for (int k = 0; k < K; ++k) softmax_fast<C, false>(z[k], st.p[k], st.l[k]);
        // Dirichlet mix + argmax (:251-255) with the runner-up, to know when the fast value can be trusted
        int y = 0;
        float best = 0.f, second = -1.f;
#pragma unroll
        for (int c = 0; c < C; ++c) {
            float mix = w[0] * st.p[0][c];
#pragma unroll
            for (int k = 1; k < K; ++k) mix = fmaf(w[k], st.p[k][c], mix);
            if (c == 0) best = mix;
            else if (mix > best) { second = best; best = mix; y = c; }
            else second = fmaxf(second, mix);
        }
        kl_terms<K, C, false, false>(st);
        // An underflowed probability (p flushed to 0 -> log2 p = -inf) always surfaces as a non-finite V:
        // q_c > 0 gives V = +inf, q_c == 0 gives 0 * -inf = NaN.  One rarely-taken branch per pixel covers
        // both slow paths: near-tie -> exact argmax; non-finite -> logs from (z - max) and xlogy's 0 rule.
        float vs = st.V[0];
#pragma unroll
        for (int k = 1; k < K; ++k) vs += st.V[k];
        const bool tie = !(best - second > kTieMargin);
        const bool bad = !(fabsf(vs) < 1e30f);
        if (__builtin_expect(tie || bad, 0)) {
            if (tie) y = argmax_exact_gmem<K, C>(a, pix_off);
            if (bad) {
#pragma unroll
                for (int k = 0; k < K; ++k) log2_softmax_underflow_fix<C>(z[k], st.l[k]);
                kl_terms<K, C, false, true>(st);
            }
        }
        st.y = y;
    }
}

// Inference form of pixel_forward (default arithmetic): softmaxes, mean prediction and KL maps as above, but the label
// is the argmax of the mean prediction q itself (UAPS_train.py:223 followed by argmax), bit-exact with torch's
// argmax(q, 1) by the same near-tie rule.  st.E is left to dead-code elimination.
template <int K, int C, typename Args>
__device__ __forceinline__ void pixel_mean_forward(const float (&z)[K][C], const Args& a, size_t pix_off, PixelState<K, C>& st) {
#pragma unroll
    for (int k = 0; k < K; ++k) softmax_fast<C, false>(z[k], st.p[k], st.l[k]);
    kl_terms<K, C, false, false>(st);
    int y = 0;
    float best = st.q[0], second = -1.f;
#pragma unroll
    for (int c = 1; c < C; ++c) {
        if (st.q[c] > best) { second = best; best = st.q[c]; y = c; }
        else second = fmaxf(second, st.q[c]);
    }
    float vs = st.V[0];
#pragma unroll
    for (int k = 1; k < K; ++k) vs += st.V[k];
    const bool tie = !(best - second > kTieMargin);
    const bool bad = !(fabsf(vs) < 1e30f);
    if (__builtin_expect(tie || bad, 0)) {
        if (tie) y = argmax_exact_gmem<K, C, true>(a, pix_off);
        if (bad) {
#pragma unroll
            for (int k = 0; k < K; ++k) log2_softmax_underflow_fix<C>(z[k], st.l[k]);
            kl_terms<K, C, false, true>(st);
        }
    }
    st.y = y;
}

// K*C independent vector loads of one pixel group (one per class plane of every decoder)
template <int K, int C, int VEC, typename Args>
__device__ __forceinline__ void load_group(const Args& a, unsigned g, float (&zv)[K][C][VEC]) {
    const unsigned b = g / a.groups_per_image;
    const unsigned hw = (g - b * a.groups_per_image) * VEC;
    const size_t base = (size_t)b * C * a.HW + hw;
#pragma unroll
    for (int k = 0; k < K; ++k)
#pragma unroll
        for (int c = 0; c < C; ++c) load_vec<VEC>(a.z[k] + base + (size_t)c * a.HW, zv[k][c]);
}

// ---- pass 1 --------------------------------------------------------------------------------
// running sums of one thread, flat in the order of `sums` (see uaps_loss_sums_count); every index
// below is a compile-time constant after unrolling, so the array lives in registers
template <int K, int C>
struct AccIdx {
    static constexpr int CE = 0, E = K, V = 2 * K, I = 3 * K, P = 3 * K + K * C, T = 3 * K + 2 * K * C;
    static constexpr int S = 3 * K + 2 * K * C + C;
};

// fold one pixel into the running sums.  The label's one-hot is applied as arithmetic masks (keeps
// p/l in registers: a select chain would be turned into a local-memory indexed load)
template <int K, int C, bool EXACT>
__device__ __forceinline__ void accumulate_pixel(const PixelState<K, C>& st, float (&acc)[AccIdx<K, C>::S]) {
    using AI = AccIdx<K, C>;
    constexpr float U = LogUnit<EXACT>::U;
    float oh[C];
#pragma unroll
    for (int c = 0; c < C; ++c) {
        oh[c] = (st.y == c) ? 1.f : 0.f;
        acc[AI::T + c] += oh[c];
    }
#pragma unroll
    for (int k = 0; k < K; ++k) {
        acc[AI::E + k] += st.E[k];
        acc[AI::V + k] += st.V[k];
        float ly = 0.f;
#pragma unroll
        for (int c = 0; c < C; ++c) {
            ly = fmaf(oh[c], st.l[k][c], ly);
            acc[AI::I + k * C + c] = fmaf(oh[c], st.p[k][c], acc[AI::I + k * C + c]);
            acc[AI::P + k * C + c] += st.p[k][c];
        }
        acc[AI::CE + k] = fmaf(-U, ly, acc[AI::CE + k]);
    }
}

// block-level reduction of the running sums into this block's column of partials[S][LOSS_MAX_BLOCKS]
template <int S, int THREADS>
__device__ __forceinline__ void block_store_partials(float (&acc)[S], float* __restrict__ partials,
                                                     float (*s_red)[S]) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int i = 0; i < S; ++i) {
        const float r = warp_sum(acc[i]);
        if (lane == 0) s_red[warp][i] = r;
    }
    __syncthreads();
    for (int i = threadIdx.x; i < S; i += THREADS) {
        float r = 0.f;
#pragma unroll
        for (int wv = 0; wv < THREADS / kWarp; ++wv) r += s_red[wv][i];
        partials[(size_t)i * LOSS_MAX_BLOCKS + blockIdx.x] = r;
    }
}

// WDEV: the mix weights come from device memory (a.w_dev, the device-resident step state) instead of the by-value
// argument block.  A template parameter, not a run-time select: by-value weights are constant-bank FMA operands and
// cost no registers, and these kernels sit exactly at their register budget (a run-time select spilled).
template <int K, int C, int VEC, bool SUP, bool EXACT, bool PF, bool WDEV>
__global__ void __launch_bounds__(LOSS_THREADS, min_ctas(K, C, PF ? 2 * VEC : VEC, true))
loss_pass1_kernel(const __grid_constant__ LossArgs a, float* __restrict__ partials) {
    constexpr int S = sums_count(K, C);
    __shared__ float s_red[LOSS_THREADS / kWarp][S];
    pdl_wait();                       // the logits may be the previous kernel's output (out_conv epilogue)
    pdl_trigger();                    // the fold kernel's CTA may take the first SM slot that frees up

    float w[K];
#pragma unroll
    for (int k = 0; k < K; ++k) w[k] = WDEV ? a.w_dev[k] : a.w[k];

    float acc[S];
#pragma unroll
    for (int i = 0; i < S; ++i) acc[i] = 0.f;

    // software pipelining (PF): the next group's K*C loads are issued before this group is computed, so
    // HBM latency overlaps the ~330 instructions/pixel instead of stalling the first consumer
    const unsigned stride = gridDim.x * LOSS_THREADS;
    unsigned g = blockIdx.x * LOSS_THREADS + threadIdx.x;
    float zn[PF ? K : 1][PF ? C : 1][PF ? VEC : 1];
    if constexpr (PF) { if (g < a.ngroups) load_group<K, C, VEC>(a, g, zn); }
    for (; g < a.ngroups; g += stride) {
        const unsigned b = g / a.groups_per_image;
        const unsigned hw = (g - b * a.groups_per_image) * VEC;
        const size_t base = (size_t)b * C * a.HW + hw;
        float zv[K][C][VEC];
        if constexpr (PF) {
#pragma unroll
            for (int k = 0; k < K; ++k)
#pragma unroll
                for (int c = 0; c < C; ++c)
#pragma unroll
                    for (int j = 0; j < VEC; ++j) zv[k][c][j] = zn[k][c][j];
            if (g + stride < a.ngroups) load_group<K, C, VEC>(a, g + stride, zn);
        } else {
            load_group<K, C, VEC>(a, g, zv);
        }
        long long lab[VEC];
        if constexpr (SUP) {
#pragma unroll
            for (int j = 0; j < VEC; ++j) lab[j] = __ldg(a.labels + (size_t)b * a.HW + hw + j);
        }
        float ev[K][VEC];
        long long yv[VEC];
#pragma unroll
        for (int j = 0; j < VEC; ++j) {
            float z[K][C];
#pragma unroll
            for (int k = 0; k < K; ++k)
#pragma unroll
                for (int c = 0; c < C; ++c) z[k][c] = zv[k][c][j];
            PixelState<K, C> st;
            pixel_forward<K, C, SUP, EXACT>(z, w, SUP ? (int)lab[j] : 0, a, base + j, st);
            yv[j] = st.y;
#pragma unroll
            for (int k = 0; k < K; ++k) ev[k][j] = st.E[k];
            accumulate_pixel<K, C, EXACT>(st, acc);
        }
        if (a.pseudo != nullptr) {
#pragma unroll
            for (int j = 0; j < VEC; ++j) a.pseudo[(size_t)b * a.HW + hw + j] = yv[j];
        }
        if (a.write_ev) {
#pragma unroll
            for (int k = 0; k < K; ++k)
                if (a.out[k] != nullptr) store_vec<VEC>(a.out[k] + (size_t)b * a.HW + hw, ev[k]);
        }
    }

    block_store_partials<S, LOSS_THREADS>(acc, partials, s_red);
}

// ---- finalize (compiled only into the entry-point unit) -----------------------------------------
#ifdef UAPS_LOSS_ENTRY
// Deterministic fp64 fold of the per-block partials [S][LOSS_MAX_BLOCKS]: one warp per sum, every
// lane's loads issued together (unrolled, predicated) so a row costs one L2 round trip.
__global__ void __launch_bounds__(256) loss_fold_kernel(const float* __restrict__ partials, int S, unsigned nblocks,
                                                        double* __restrict__ sums) {
    pdl_trigger();
    pdl_wait();
    const int lane = threadIdx.x & 31;
    const int i = blockIdx.x * (256 / kWarp) + (threadIdx.x >> 5);
    if (i >= S) return;
    const float* row = partials + (size_t)i * LOSS_MAX_BLOCKS;
    float v[LOSS_MAX_BLOCKS / kWarp];
#pragma unroll
    for (int u = 0; u < LOSS_MAX_BLOCKS / kWarp; ++u) {
        const unsigned blk = u * kWarp + lane;
        v[u] = (blk < nblocks) ? __ldcg(row + blk) : 0.f;
    }
    double r = 0.0;
#pragma unroll
    for (int u = 0; u < LOSS_MAX_BLOCKS / kWarp; ++u) r += (double)v[u];
    r = warp_sum(r);
    if (lane == 0) sums[i] = r;
}

// One CTA of 1024 threads folds partials[S][LOSS_MAX_BLOCKS] into s_sums[S] (fp64): a HALF-warp per sum row, so the
// up-to-64 rows go in one pass; every lane's loads are issued together (unrolled, predicated), the adds run in a fixed
// order (deterministic).  Ends with __syncthreads().
__device__ __forceinline__ void cta_fold_rows(const float* __restrict__ partials, int S, unsigned nblocks, double* s_sums) {
    constexpr int HALF = 16, PER_LANE = LOSS_MAX_BLOCKS / HALF;
    const int sub = threadIdx.x & (HALF - 1);
    for (int base = (threadIdx.x >> 5) * 2; base < S; base += 2 * (1024 / 32)) {    // warp-uniform trip count (S may be odd)
        const int i = base + ((threadIdx.x >> 4) & 1);
        const bool live = i < S;
        const float* row = partials + (size_t)(live ? i : 0) * LOSS_MAX_BLOCKS;
        float v[PER_LANE];
#pragma unroll
        for (int u = 0; u < PER_LANE; ++u) {
            const unsigned blk = u * HALF + sub;
            v[u] = (live && blk < nblocks) ? __ldcg(row + blk) : 0.f;
        }
        double r = 0.0;
#pragma unroll
        for (int u = 0; u < PER_LANE; ++u) r += (double)v[u];
#pragma unroll
        for (int o = HALF / 2; o > 0; o >>= 1) r += __shfl_xor_sync(0xffffffffu, r, o);
        if (live && sub == 0) s_sums[i] = r;
    }
    __syncthreads();
}

// Cooperative finalize (whole CTA, >= K*C threads): the K*C fp64 divisions of the Dice terms run in parallel, thread 0
// combines them in the same order as finalize_from_sums.  s_term: K*C doubles of shared memory.
__device__ __forceinline__ void cta_finalize(const double* sums, int K, int C, double N, float cw1, float cw2, int supervised,
                                             float* sc, double* s_term) {
    const double* sI = sums + 3 * K;
    const double* sP = sums + 3 * K + K * C;
    const double* sT = sums + 3 * K + 2 * K * C;
    float* Ikc = sc + UAPS_SC_BASE + 4 * K;
    float* Card = Ikc + K * C;
    const int t = threadIdx.x;
    if (t < K * C) {
        const double card = sP[t] + sT[t % C];
        s_term[t] = 2.0 * sI[t] / (card + 1e-7);                          // pytorch_losses.py:88
        Ikc[t] = (float)sI[t];
        Card[t] = (float)card;
    }
    __syncthreads();
    if (t != 0) return;
    const double* sCE = sums;
    const double* sE = sums + K;
    const double* sV = sums + 2 * K;
    float* ps = sc + UAPS_SC_BASE;
    float* Eb = ps + K;
    float* CE = Eb + K;
    float* DI = CE + K;
    const double invN = 1.0 / N;
    double ps_loss = 0.0, unc = 0.0, mce = 0.0, mdi = 0.0;
    for (int k = 0; k < K; ++k) {
        const double ce = sCE[k] / N;
        double d = 0.0;
        for (int c = 0; c < C; ++c) d += s_term[k * C + c];
        const double dice = 1.0 - d / C;
        const double psk = 0.5 * (ce + dice);                          // UAPS_train.py:259-262
        const double eb = supervised ? 1.0 : sE[k] / N;
        ps[k] = (float)psk; Eb[k] = (float)eb; CE[k] = (float)ce; DI[k] = (float)dice;
        ps_loss += psk * eb;                                           // :265-268 (scalar x mean(E))
        unc += sV[k] / N;
        mce += (double)(float)ce; mdi += (double)(float)dice;
    }
    ps_loss /= K;                                                       // :277
    unc /= K;                                                           // :241-243
    sc[UAPS_SC_PS_LOSS] = (float)ps_loss;
    sc[UAPS_SC_L_UNCERT] = supervised ? 0.f : (float)unc;
    sc[UAPS_SC_LOSS_U] = supervised ? (float)ps_loss : (float)((double)cw1 * ps_loss + (double)cw2 * unc);
    sc[UAPS_SC_CW1] = supervised ? 1.f : cw1;
    sc[UAPS_SC_CW2] = supervised ? 0.f : cw2;
    sc[UAPS_SC_INV_N] = (float)invN;
    sc[UAPS_SC_MEAN_CE] = (float)(mce / K);                             // :216 total_loss_ce
    sc[UAPS_SC_MEAN_DICE] = (float)(mdi / K);                           // :217 total_loss_dice
}

// Single-rank fast path: fold + finalize in one launch (one CTA of 32 warps, a warp per sum row, then thread 0
// turns the sums into the scalars).  Saves a kernel and a launch gap per step versus fold -> finalize.
__device__ void finalize_from_sums(const double* sums, int K, int C, double N, float cw1, float cw2, int supervised, float* sc);

__global__ void __launch_bounds__(1024) loss_fold_finalize_kernel(const float* __restrict__ partials, int S, unsigned nblocks,
                                                                   double* __restrict__ sums, int K, int C, double N, float cw1,
                                                                   float cw2, int supervised, float* __restrict__ sc,
                                                                   const float* __restrict__ wcw_dev) {
    __shared__ double s_sums[3 * KMAX + 2 * KMAX * CMAX + CMAX];
    __shared__ double s_term[KMAX * CMAX];
    pdl_trigger();                    // pass 2 may start prefetching its logits now; it waits for THIS kernel before using sc
    pdl_wait();                       // partials of pass 1
    cta_fold_rows(partials, S, nblocks, s_sums);
    if (threadIdx.x < S) sums[threadIdx.x] = s_sums[threadIdx.x];
    if (wcw_dev != nullptr) { cw1 = wcw_dev[UAPS_WCW_CW1]; cw2 = wcw_dev[UAPS_WCW_CW2]; }
    cta_finalize(s_sums, K, C, N, cw1, cw2, supervised, sc, s_term);
}

__device__ void finalize_from_sums(const double* sums, int K, int C, double N, float cw1, float cw2, int supervised, float* sc) {
    const double* sCE = sums;
    const double* sE = sums + K;
    const double* sV = sums + 2 * K;
    const double* sI = sums + 3 * K;
    const double* sP = sums + 3 * K + K * C;
    const double* sT = sums + 3 * K + 2 * K * C;
    float* ps = sc + UAPS_SC_BASE;
    float* Eb = ps + K;
    float* CE = Eb + K;
    float* DI = CE + K;
    float* Ikc = DI + K;
    float* Card = Ikc + K * C;
    double ps_loss = 0.0, unc = 0.0;
    for (int k = 0; k < K; ++k) {
        const double ce = sCE[k] / N;
        double d = 0.0;
        for (int c = 0; c < C; ++c) {
            const double card = sP[k * C + c] + sT[c];
            d += 2.0 * sI[k * C + c] / (card + 1e-7);                 // pytorch_losses.py:88
            Ikc[k * C + c] = (float)sI[k * C + c];
            Card[k * C + c] = (float)card;
        }
        const double dice = 1.0 - d / C;
        const double psk = 0.5 * (ce + dice);                          // UAPS_train.py:259-262
        const double eb = supervised ? 1.0 : sE[k] / N;
        ps[k] = (float)psk; Eb[k] = (float)eb; CE[k] = (float)ce; DI[k] = (float)dice;
        ps_loss += psk * eb;                                           // :265-268 (scalar x mean(E))
        unc += sV[k] / N;
    }
    ps_loss /= K;                                                       // :277
    unc /= K;                                                           // :241-243
    sc[UAPS_SC_PS_LOSS] = (float)ps_loss;
    sc[UAPS_SC_L_UNCERT] = supervised ? 0.f : (float)unc;
    sc[UAPS_SC_LOSS_U] = supervised ? (float)ps_loss : (float)((double)cw1 * ps_loss + (double)cw2 * unc);
    sc[UAPS_SC_CW1] = supervised ? 1.f : cw1;
    sc[UAPS_SC_CW2] = supervised ? 0.f : cw2;
    sc[UAPS_SC_INV_N] = (float)(1.0 / N);
    double mce = 0.0, mdi = 0.0;
    for (int k = 0; k < K; ++k) { mce += CE[k]; mdi += DI[k]; }
    sc[UAPS_SC_MEAN_CE] = (float)(mce / K);                             // :216 total_loss_ce
    sc[UAPS_SC_MEAN_DICE] = (float)(mdi / K);                           // :217 total_loss_dice
}

__global__ void loss_finalize_kernel(const double* __restrict__ sums, int K, int C, double N,
                                     float cw1, float cw2, int supervised, float* __restrict__ sc) {
    pdl_trigger();
    pdl_wait();
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    finalize_from_sums(sums, K, C, N, cw1, cw2, supervised, sc);
}
#endif  // UAPS_LOSS_ENTRY

// ---- pass 2 --------------------------------------------------------------------------------
template <int K, int C>
struct GradConsts {
    float psk[K];        // ps_k
    float cce[K];        // (d loss / d CE_k) / N
    float A[K][C];       // -(d loss / d Dice_k) * (2/C) / (Card + eps)
    float Bc[K][C];      // +(d loss / d Dice_k) * (2/C) * I / (Card + eps)^2
    float lam1, lam2, invNK;
};

// one thread turns the loss scalars and the upstream gradient vector into the per-(k,c) constants
template <int K, int C>
__device__ __forceinline__ void load_grad_consts(GradConsts<K, C>& gc, const float* __restrict__ sc,
                                                 const float* __restrict__ grad_out) {
    // upstream gradient vector, laid out like scalars[] (only the five differentiable slots are read)
    const float g_loss = grad_out[UAPS_SC_LOSS_U], g_ps = grad_out[UAPS_SC_PS_LOSS], g_unc = grad_out[UAPS_SC_L_UNCERT];
    const float g_ce = grad_out[UAPS_SC_MEAN_CE], g_dice = grad_out[UAPS_SC_MEAN_DICE];
    const float lam1 = g_loss * sc[UAPS_SC_CW1] + g_ps;
    const float lam2 = g_loss * sc[UAPS_SC_CW2] + g_unc;
    const float invN = sc[UAPS_SC_INV_N];
    const float* ps = sc + UAPS_SC_BASE;
    const float* Eb = ps + K;
    const float* Ikc = ps + 4 * K;
    const float* Card = Ikc + K * C;
    gc.lam1 = lam1; gc.lam2 = lam2; gc.invNK = invN / K;
    for (int k = 0; k < K; ++k) {
        gc.psk[k] = ps[k];
        const float half = lam1 * Eb[k] / (2.f * K);           // d loss / d ps_k * 0.5
        const float dce = half + g_ce / K;                     // d loss / d CE_k
        const float ddice = half + g_dice / K;                 // d loss / d Dice_k
        gc.cce[k] = dce * invN;
        for (int c = 0; c < C; ++c) {
            const float den = Card[k * C + c] + 1e-7f;
            gc.A[k][c] = -ddice * (2.f / C) / den;
            gc.Bc[k][c] = ddice * (2.f / C) * Ikc[k * C + c] / (den * den);
        }
    }
}

// d loss / d z for one pixel (SURVEY.md 8 a16; closed form checked against autograd in oracle/)
template <int K, int C, bool SUP, bool EXACT>
__device__ __forceinline__ void pixel_backward(const PixelState<K, C>& st, const GradConsts<K, C>& gc,
                                               float (&dz)[K][C]) {
    float gk[K];
    float Gq[C];
#pragma unroll
    for (int c = 0; c < C; ++c) Gq[c] = 0.f;
    if constexpr (!SUP) {
#pragma unroll
        for (int k = 0; k < K; ++k) {
            gk[k] = (gc.lam2 - gc.lam1 * gc.psk[k] * st.E[k]) * gc.invNK;
#pragma unroll
            for (int c = 0; c < C; ++c) Gq[c] += gk[k] * fmaf(LogUnit<EXACT>::U, st.lq[c] - st.l[k][c], 1.f);
        }
#pragma unroll
        for (int c = 0; c < C; ++c) Gq[c] *= (1.0f / K);
    }
    float oh[C];
#pragma unroll
    for (int c = 0; c < C; ++c) oh[c] = (st.y == c) ? 1.f : 0.f;
#pragma unroll
    for (int k = 0; k < K; ++k) {
        float Gl[C], Gp[C];
        float sGl = 0.f, dot = 0.f;
#pragma unroll
        for (int c = 0; c < C; ++c) {
            float gl = -gc.cce[k] * oh[c];
            if constexpr (!SUP) gl = fmaf(-gk[k], st.q[c], gl);
            const float gp = fmaf(gc.A[k][c], oh[c], Gq[c] + gc.Bc[k][c]);
            Gl[c] = gl; Gp[c] = gp;
            sGl += gl;
            dot = fmaf(st.p[k][c], gp, dot);
        }
#pragma unroll
        for (int c = 0; c < C; ++c) dz[k][c] = fmaf(st.p[k][c], (Gp[c] - dot) - sGl, Gl[c]);
    }
}

template <int K, int C, int VEC, bool SUP, bool EXACT, bool PF, bool WDEV>
__global__ void __launch_bounds__(LOSS_THREADS, min_ctas(K, C, PF ? 2 * VEC : VEC, false))
loss_pass2_kernel(const __grid_constant__ LossArgs a, const float* __restrict__ sc, const float* __restrict__ grad_out) {
    __shared__ GradConsts<K, C> gc;

    float w[K];
#pragma unroll
    for (int k = 0; k < K; ++k) w[k] = WDEV ? a.w_dev[k] : a.w[k];

    // software pipelining (PF): the next group's K*C loads are issued before this group is computed, so
    // HBM latency overlaps the ~330 instructions/pixel instead of stalling the first consumer
    const unsigned stride = gridDim.x * LOSS_THREADS;
    unsigned g = blockIdx.x * LOSS_THREADS + threadIdx.x;
    float zn[PF ? K : 1][PF ? C : 1][PF ? VEC : 1];
    if constexpr (PF) { if (g < a.ngroups) load_group<K, C, VEC>(a, g, zn); }     // in flight while the predecessor drains
    pdl_wait();                       // scalars (fold/finalize), upstream gradient, labels
    pdl_trigger();
    if (threadIdx.x == 0) load_grad_consts<K, C>(gc, sc, grad_out);
    __syncthreads();
    for (; g < a.ngroups; g += stride) {
        const unsigned b = g / a.groups_per_image;
        const unsigned hw = (g - b * a.groups_per_image) * VEC;
        const size_t base = (size_t)b * C * a.HW + hw;
        float zv[K][C][VEC];
        if constexpr (PF) {
#pragma unroll
            for (int k = 0; k < K; ++k)
#pragma unroll
                for (int c = 0; c < C; ++c)
#pragma unroll
                    for (int j = 0; j < VEC; ++j) zv[k][c][j] = zn[k][c][j];
            if (g + stride < a.ngroups) load_group<K, C, VEC>(a, g + stride, zn);
        } else {
            load_group<K, C, VEC>(a, g, zv);
        }
        long long lab[VEC];
        if constexpr (SUP) {
#pragma unroll
            for (int j = 0; j < VEC; ++j) lab[j] = __ldg(a.labels + (size_t)b * a.HW + hw + j);
        }
#pragma unroll
        for (int j = 0; j < VEC; ++j) {
            float z[K][C];
#pragma unroll
            for (int k = 0; k < K; ++k)
#pragma unroll
                for (int c = 0; c < C; ++c) z[k][c] = zv[k][c][j];
            PixelState<K, C> st;
            pixel_forward<K, C, SUP, EXACT>(z, w, SUP ? (int)lab[j] : 0, a, base + j, st);
            float dz[K][C];
            pixel_backward<K, C, SUP, EXACT>(st, gc, dz);
#pragma unroll
            for (int k = 0; k < K; ++k)
#pragma unroll
                for (int c = 0; c < C; ++c) zv[k][c][j] = dz[k][c];
        }
#pragma unroll
        for (int k = 0; k < K; ++k)
#pragma unroll
            for (int c = 0; c < C; ++c) store_vec<VEC>(a.out[k] + base + (size_t)c * a.HW, zv[k][c]);
    }
}

// ---- per-K launchers (one translation unit per K keeps nvcc parallel and compile time bounded) ---
// Kernel variants.  Measured on B200 (profiles/r01_loss_variants.txt): software-pipelined register
// kernels beat both the plain ones (first-use stall on the K*C loads was 36% of all warp stall
// samples) and a cp.async.bulk/mbarrier shared-memory ring (which removed that stall but lost the
// cross-pixel ILP the per-thread vector gives); pass 1 likes 4 pixels/thread, pass 2 two.
enum LossImpl { IMPL_VEC4_PF = 0, IMPL_VEC2_PF = 1, IMPL_SCALAR = 2, IMPL_EXACT = 3, IMPL_VEC2 = 4, IMPL_VEC4 = 5 };

__host__ __device__ constexpr bool has_vec4(int K, int C) { return K * C <= 16; }
__host__ __device__ constexpr bool has_vec2(int K, int C) { return K * C <= 24; }

template <typename Kern>
inline int grid_for(Kern kern, unsigned ngroups) {
    int occ = 1;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, LOSS_THREADS, 0) != cudaSuccess || occ < 1) occ = 1;
    long long want = ceil_div<long long>(ngroups, LOSS_THREADS);
    long long cap = (long long)device_info().sm_count * occ;
    if (cap > LOSS_MAX_BLOCKS) cap = LOSS_MAX_BLOCKS;
    return (int)(want < cap ? want : cap);
}

template <int K, int C, int VEC, bool SUP, bool EXACT, bool PF, bool WDEV>
inline int launch_reg(bool pass2, LossArgs a, float* partials, const float* sc, const float* go, int* nblocks,
                      cudaStream_t st) {
    a.groups_per_image = (unsigned)(a.HW / VEC);
    a.ngroups = (unsigned)a.B * a.groups_per_image;
    if (!pass2) {
        auto kern = loss_pass1_kernel<K, C, VEC, SUP, EXACT, PF, WDEV>;
        static const int grid_cap = grid_for(kern, 0x7fffffffu);       // occupancy query once per instantiation
        const long long want = ceil_div<long long>(a.ngroups, LOSS_THREADS);
        *nblocks = (int)(want < grid_cap ? want : grid_cap);
        const cudaError_t e = launch_pdl(kern, dim3(*nblocks), dim3(LOSS_THREADS), st, pdl_enabled(), a, partials);
        if (e != cudaSuccess) return (int)e;
    } else {
        auto kern = loss_pass2_kernel<K, C, VEC, SUP, EXACT, PF, WDEV>;
        static const int grid_cap = grid_for(kern, 0x7fffffffu);
        const long long want = ceil_div<long long>(a.ngroups, LOSS_THREADS);
        *nblocks = (int)(want < grid_cap ? want : grid_cap);
        const cudaError_t e = launch_pdl(kern, dim3(*nblocks), dim3(LOSS_THREADS), st, pdl_enabled(), a, sc, go);
        if (e != cudaSuccess) return (int)e;
    }
    UAPS_LAUNCH_CHECK();
    return UAPS_OK;
}

template <int K, int C>
inline int launch_kc(int impl, bool sup, bool pass2, const LossArgs& a, float* partials, const float* sc,
                     const float* go, int* nblocks, cudaStream_t st) {
#define UAPS_RUN(VEC, EXACT, PF)                                                                       \
    (sup ? launch_reg<K, C, VEC, true, EXACT, PF, false>(pass2, a, partials, sc, go, nblocks, st)                      \
         : (a.w_dev != nullptr ? launch_reg<K, C, VEC, false, EXACT, PF, true>(pass2, a, partials, sc, go, nblocks, st) \
                               : launch_reg<K, C, VEC, false, EXACT, PF, false>(pass2, a, partials, sc, go, nblocks, st)))
    if (impl == IMPL_EXACT) return UAPS_RUN(1, true, false);
#ifdef UAPS_LOSS_EXTRA_VARIANTS       // tuning builds only: vector kernels WITHOUT the register prefetch (3 CTAs per SM instead of 2).
    // Measured on B200, K=4 C=4 64x256x256, pass 1 + fold: VEC4+prefetch (default, 2 CTAs/SM) 82.1 us | VEC2 no prefetch 93.3 |
    // VEC2+prefetch 108.2 | VEC4 no prefetch (spills) 108.9 | scalar 114.7 -- more resident warps do not help: the kernel
    // needs the 4-pixel instruction-level parallelism inside a thread, not thread-level parallelism.
    if constexpr (has_vec2(K, C)) { if (impl == IMPL_VEC2) return UAPS_RUN(2, false, false); }
    if constexpr (has_vec4(K, C)) { if (impl == IMPL_VEC4) return UAPS_RUN(4, false, false); }
#endif
    if constexpr (has_vec4(K, C)) { if (impl == IMPL_VEC4_PF) return UAPS_RUN(4, false, true); }
    if constexpr (has_vec2(K, C)) { if (impl == IMPL_VEC4_PF || impl == IMPL_VEC2_PF) return UAPS_RUN(2, false, true); }
    return UAPS_RUN(1, false, false);
#undef UAPS_RUN
}

template <int K>
int launch_loss_k(int C, int impl, bool sup, bool pass2, const LossArgs& a, float* partials, const float* sc,
                  const float* go, int* nblocks, cudaStream_t st) {
    switch (C) {
        case 2: return launch_kc<K, 2>(impl, sup, pass2, a, partials, sc, go, nblocks, st);
        case 3: return launch_kc<K, 3>(impl, sup, pass2, a, partials, sc, go, nblocks, st);
        case 4: return launch_kc<K, 4>(impl, sup, pass2, a, partials, sc, go, nblocks, st);
        case 5: return launch_kc<K, 5>(impl, sup, pass2, a, partials, sc, go, nblocks, st);
        case 6: return launch_kc<K, 6>(impl, sup, pass2, a, partials, sc, go, nblocks, st);
        case 7: return launch_kc<K, 7>(impl, sup, pass2, a, partials, sc, go, nblocks, st);
        case 8: return launch_kc<K, 8>(impl, sup, pass2, a, partials, sc, go, nblocks, st);
    }
    return UAPS_ERANGE;
}

}  // namespace loss
}  // namespace uaps
