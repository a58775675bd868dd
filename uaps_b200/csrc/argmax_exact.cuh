// pred = argmax(softmax(logits)) exactly as torch computes it, shared by the confusion matrix (metrics.cu) and the
// validation head (val_head.cu): softmax rounding can merge two nearly equal logits into a tie that argmax then resolves
// to the lower index, so the softmax chain is reproduced.
#pragma once
#include "common.cuh"

namespace uaps {

template <int C>
__device__ __forceinline__ int argmax_softmax(const float (&z)[C]) {
    float m = z[0];
#pragma unroll
    for (int c = 1; c < C; ++c) m = fmaxf(m, z[c]);
    float e[C], s = 0.f;
#pragma unroll
    for (int c = 0; c < C; ++c) { e[c] = expf(__fsub_rn(z[c], m)); s = __fadd_rn(s, e[c]); }
    int y = 0;
    float best = __fdiv_rn(e[0], s);
#pragma unroll
    for (int c = 1; c < C; ++c) {
        const float p = __fdiv_rn(e[c], s);
        if (p > best) { best = p; y = c; }
    }
    return y;
}

}  // namespace uaps
