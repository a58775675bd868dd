// On-device segmentation metrics (SURVEY.md 8(f2)): the confusion matrix behind utilities/metrics.py
// (pixel_accuracy :8-13, mIoU :16-37, mDice :40-61) in one pass over the logits, so the training loop needs one
// host sync per epoch instead of the reference's ~20 per iteration (UAPS_train.py:295-306).
// pred = argmax(softmax(logits)) exactly as torch computes it (argmax_exact.cuh, shared with the validation head).
#include "argmax_exact.cuh"

namespace uaps {
namespace {

constexpr int MT = 256;

// conf[label][pred] += 1 for every pixel; labels outside [0, C) are ignored
template <int C>
__global__ void __launch_bounds__(MT) confusion_kernel(const float* __restrict__ logits, const long long* __restrict__ labels,
                                                       int B, long long HW, unsigned long long* __restrict__ conf) {
    __shared__ unsigned int s_conf[C * C];
    for (int i = threadIdx.x; i < C * C; i += MT) s_conf[i] = 0u;
    __syncthreads();
    const long long total = (long long)B * HW;
    for (long long n = (long long)blockIdx.x * MT + threadIdx.x; n < total; n += (long long)gridDim.x * MT) {
        const long long b = n / HW, hw = n - b * HW;
        float z[C];
#pragma unroll
        for (int c = 0; c < C; ++c) z[c] = __ldg(logits + ((size_t)b * C + c) * HW + hw);
        const long long lab = __ldg(labels + n);
        if (lab >= 0 && lab < C) atomicAdd(&s_conf[(int)lab * C + argmax_softmax<C>(z)], 1u);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < C * C; i += MT)
        if (s_conf[i] != 0u) atomicAdd(conf + i, (unsigned long long)s_conf[i]);
}

}  // namespace
}  // namespace uaps

using namespace uaps;

// logits: [B,C,HW] fp32 NCHW; labels: [B,HW] int64; conf: C*C uint64 counters, ACCUMULATED into (row = label, col = prediction)
UAPS_API int uaps_confusion(const float* logits, const int64_t* labels, int B, int C, int64_t HW, uint64_t* conf,
                            cudaStream_t stream) {
    if (logits == nullptr || labels == nullptr || conf == nullptr || B <= 0 || HW <= 0) return UAPS_EINVAL;
    if (C < 2 || C > UAPS_CMAX) return UAPS_ERANGE;
    if (!aligned_to(logits, 4) || !aligned_to(labels, 8) || !aligned_to(conf, 8)) return UAPS_EALIGN;
    const long long total = (long long)B * HW;
    long long want = ceil_div<long long>(total, MT), cap = (long long)device_info().sm_count * 8;
    const int grid = (int)(want < cap ? want : cap);
    const long long* lab = reinterpret_cast<const long long*>(labels);
    unsigned long long* cf = reinterpret_cast<unsigned long long*>(conf);
    switch (C) {
        case 2: confusion_kernel<2><<<grid, MT, 0, stream>>>(logits, lab, B, HW, cf); break;
        case 3: confusion_kernel<3><<<grid, MT, 0, stream>>>(logits, lab, B, HW, cf); break;
        case 4: confusion_kernel<4><<<grid, MT, 0, stream>>>(logits, lab, B, HW, cf); break;
        case 5: confusion_kernel<5><<<grid, MT, 0, stream>>>(logits, lab, B, HW, cf); break;
        case 6: confusion_kernel<6><<<grid, MT, 0, stream>>>(logits, lab, B, HW, cf); break;
        case 7: confusion_kernel<7><<<grid, MT, 0, stream>>>(logits, lab, B, HW, cf); break;
        case 8: confusion_kernel<8><<<grid, MT, 0, stream>>>(logits, lab, B, HW, cf); break;
    }
    UAPS_LAUNCH_CHECK();
    return UAPS_OK;
}
