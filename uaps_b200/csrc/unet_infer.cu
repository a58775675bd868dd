// Whole-network inference through the C ABI: the eval-mode forward of UNet_UAPS's encoder + main decoder
// (UAPS_unet.py:224-226, the output UAPS_train.py:377 and UAPS-Testing.ipynb keep), without PyTorch.
//
// uaps_unet_infer_prepare folds every BatchNorm's running statistics into the convolution in front of it (one kernel,
// the arithmetic of UNet_UAPS._fold_bn) and packs the 23 layers with one uaps_conv_pack_run launch; uaps_unet_infer_run
// is UNet_UAPS.predict's folded forward -- the entry conversion, 23 conv launches with LeakyReLU in the epilogue, 4
// max-pools, 4 upsamples, through the same entry points with the same arguments and in the same order -- plus an
// optional label map from the exact argmax of the softmax.  See include/uaps_b200.h for the contract, DESIGN.md f7.
#include <cstring>
#include <vector>

#include "argmax_exact.cuh"

namespace uaps {
namespace infer {

constexpr int kLayers = 23;                       // 5 encoder blocks x 2, 4 x (conv1x1 + 2), out_conv
constexpr int kFt[5] = {16, 32, 64, 128, 256};    // UAPS_unet.py:212
constexpr float kBnEps = 1e-5f;                   // nn.BatchNorm2d's default; eps is not part of the state_dict
constexpr float kSlope = 0.01f;                   // nn.LeakyReLU() default (:39)
constexpr int kJobBytesMax = 96;                  // capacity per uaps_conv_pack_job_bytes() record in the fold kernel's arguments
constexpr size_t kAlign = 256;

inline size_t align_up(size_t v) { return (v + kAlign - 1) / kAlign * kAlign; }

struct Layer {
    int cout, cin1, cin2, ks, bn;
    size_t src;                    // blob offset (floats) of the conv weight; bias and BN tensors follow it
    size_t w_off, b_off, p_off;    // state offsets (bytes): folded fp32 weight, folded fp32 bias, packed weights
    size_t p_bytes;
};

struct Net {
    Layer l[kLayers];
    size_t params;                 // floats in the blob
    size_t table_off;              // state offset of the pack-job table
    size_t state_bytes;
};

inline bool valid_net(int in_chns, int C) { return in_chns >= 1 && in_chns <= 16 && C >= 2 && C <= UAPS_CMAX; }

// Layers in UNet_UAPS._main_plan order, which is also state_dict order: per conv its weight and bias, then -- for the
// convs of a ConvBlock -- the BatchNorm's weight, bias, running_mean and running_var.
inline Net make_net(int in_chns, int C) {
    Net n{};
    size_t src = 0, st = align_up((size_t)kLayers * kJobBytesMax);
    int k = 0;
    auto add = [&](int cout, int cin1, int cin2, int ks, int bn) {
        Layer& L = n.l[k++];
        L.cout = cout; L.cin1 = cin1; L.cin2 = cin2; L.ks = ks; L.bn = bn;
        const size_t wn = (size_t)cout * (cin1 + cin2) * ks * ks;
        L.src = src;
        src += wn + cout + (bn ? 4 * (size_t)cout : 0);
        L.w_off = st; st = align_up(st + wn * sizeof(float));
        L.b_off = st; st = align_up(st + (size_t)cout * sizeof(float));
        L.p_bytes = uaps_conv_packed_bytes(cout, cin1, cin2, ks, 1);
        L.p_off = st; st = align_up(st + L.p_bytes);
    };
    for (int lvl = 0; lvl < 5; ++lvl) {                               // encoder.in_conv, encoder.down1..4
        add(kFt[lvl], lvl ? kFt[lvl - 1] : in_chns, 0, 3, 1);
        add(kFt[lvl], kFt[lvl], 0, 3, 1);
    }
    for (int i = 1; i <= 4; ++i) {                                    // main_decoder.up1..4: conv1x1, conv (concat)
        const int c1 = kFt[5 - i], c2 = kFt[4 - i];
        add(c2, c1, 0, 1, 0);
        add(c2, c2, c2, 3, 1);
        add(c2, c2, 0, 3, 1);
    }
    add(C, kFt[0], 0, 3, 0);                                          // main_decoder.out_conv
    n.params = src;
    n.table_off = 0;
    n.state_bytes = st;
    return n;
}

// ---- prepare: BN folding ---------------------------------------------------------------------------------------------
struct FoldLayer {
    long long src, w_dst, b_dst;   // blob offset (floats); state offsets (bytes)
    long long first;               // first element of this layer in the launch's index space (weights, then biases)
    int cout, per_co, bn;
};
struct FoldArgs {
    const float* params;
    unsigned char* state;
    FoldLayer l[kLayers];
    long long total;
    int table_words;
    uint32_t table[kLayers * kJobBytesMax / 4];    // the host-built pack table, stored into the state by block 0
};

// w' = w * s, b' = (b - mean) * s + beta with s = gamma * rsqrt(var + eps): the ops and roundings of
// UNet_UAPS._fold_bn (torch's CUDA rsqrt is rsqrtf); layers without a BatchNorm are copied.
__global__ void __launch_bounds__(256) fold_bn_kernel(const __grid_constant__ FoldArgs a) {
    grid_dep_launch();
    grid_dep_wait();
    if (blockIdx.x == 0)
        for (int i = threadIdx.x; i < a.table_words; i += blockDim.x)
            reinterpret_cast<uint32_t*>(a.state)[i] = a.table[i];
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < a.total; e += (long long)gridDim.x * blockDim.x) {
        int L = 0;
        while (L + 1 < kLayers && e >= a.l[L + 1].first) ++L;
        const FoldLayer& f = a.l[L];
        const long long k = e - f.first, wn = (long long)f.cout * f.per_co;
        const float* p = a.params + f.src;
        const int co = (int)(k < wn ? k / f.per_co : k - wn);
        float s = 1.f;
        if (f.bn) {
            const float* bn = p + wn + f.cout;                        // gamma | beta | running_mean | running_var
            s = __fmul_rn(bn[co], rsqrtf(__fadd_rn(bn[3 * f.cout + co], kBnEps)));
        }
        if (k < wn) {
            const float v = p[k];
            reinterpret_cast<float*>(a.state + f.w_dst)[k] = f.bn ? __fmul_rn(v, s) : v;
        } else {
            const float b = p[wn + co];
            const float* bn = p + wn + f.cout;
            reinterpret_cast<float*>(a.state + f.b_dst)[co] =
                f.bn ? __fadd_rn(__fmul_rn(__fsub_rn(b, bn[2 * f.cout + co]), s), bn[f.cout + co]) : b;
        }
    }
}

// ---- run: label map ----------------------------------------------------------------------------------------------------
constexpr int LABEL_THREADS = 256;

// labels[b, hw] = argmax(softmax(logits[b, :, hw])), 4 pixels per thread (HW is a multiple of 256)
template <int C>
__global__ void __launch_bounds__(LABEL_THREADS) labels_kernel(const float* __restrict__ z, uchar4* __restrict__ labels, int HW) {
    grid_dep_launch();
    grid_dep_wait();
    const int g = blockIdx.x * LABEL_THREADS + threadIdx.x;
    if (4 * g >= HW) return;
    const size_t base = (size_t)blockIdx.y * C * HW + 4 * (size_t)g;
    float zv[C][4];
#pragma unroll
    for (int c = 0; c < C; ++c) load_vec<4>(z + base + (size_t)c * HW, zv[c]);
    unsigned char y[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        float v[C];
#pragma unroll
        for (int c = 0; c < C; ++c) v[c] = zv[c][j];
        y[j] = (unsigned char)argmax_softmax<C>(v);
    }
    labels[(size_t)blockIdx.y * (HW / 4) + g] = make_uchar4(y[0], y[1], y[2], y[3]);
}

template <int C>
int launch_labels(const float* z, uint8_t* labels, int B, int HW, cudaStream_t st) {
    UAPS_LAUNCH(labels_kernel<C>, dim3(ceil_div(HW / 4, LABEL_THREADS), B), dim3(LABEL_THREADS), 0, st, z,
                reinterpret_cast<uchar4*>(labels), HW);
    return UAPS_OK;
}

// workspace: the five encoder feature maps, then two scratch buffers of the largest activation (B*H*W*16 bf16 -- the
// entry tensor, every level-0 map; the fp32 logits when the caller passes none fit too, C <= 8)
struct Ws { size_t feat[5], a, b, bytes; };
inline Ws ws_layout(int B, int H, int W) {
    Ws w{};
    size_t off = 0;
    for (int l = 0; l < 5; ++l) {
        w.feat[l] = off;
        off = align_up(off + (size_t)B * (H >> l) * (W >> l) * kFt[l] * 2);
    }
    const size_t big = align_up((size_t)B * H * W * 16 * 2);
    w.a = off; w.b = off + big; w.bytes = off + 2 * big;
    return w;
}

inline int check_shape(int B, int H, int W) {
    if (B <= 0 || H <= 0 || W <= 0) return UAPS_EINVAL;
    if (H % 16 || W % 16) return UAPS_ERANGE;                          // four 2x poolings
    if (B > 65535 || (long long)B * H * W >= (1LL << 31)) return UAPS_ERANGE;
    return UAPS_OK;
}

}  // namespace infer
}  // namespace uaps

using namespace uaps;
using namespace uaps::infer;

UAPS_API size_t uaps_unet_params_count(int in_chns, int C) {
    return valid_net(in_chns, C) ? make_net(in_chns, C).params : 0;
}

UAPS_API size_t uaps_unet_infer_state_bytes(int in_chns, int C) {
    return valid_net(in_chns, C) ? make_net(in_chns, C).state_bytes : 0;
}

UAPS_API int uaps_unet_infer_layer(int in_chns, int C, int layer, size_t* weight_offset, size_t* bias_offset,
                                   size_t* packed_offset, size_t* packed_bytes) {
    if (weight_offset == nullptr || bias_offset == nullptr || packed_offset == nullptr || packed_bytes == nullptr) return UAPS_EINVAL;
    if (!valid_net(in_chns, C) || layer < 0 || layer >= kLayers) return UAPS_ERANGE;
    const Layer& L = make_net(in_chns, C).l[layer];
    *weight_offset = L.w_off; *bias_offset = L.b_off; *packed_offset = L.p_off; *packed_bytes = L.p_bytes;
    return UAPS_OK;
}

UAPS_API size_t uaps_unet_infer_workspace_bytes(int in_chns, int C, int B, int H, int W) {
    if (!valid_net(in_chns, C) || check_shape(B, H, W) != UAPS_OK) return 0;
    return ws_layout(B, H, W).bytes;
}

UAPS_API int uaps_unet_infer_prepare(const float* params, int in_chns, int C, void* state, size_t state_bytes,
                                     cudaStream_t stream) {
    if (params == nullptr || state == nullptr) return UAPS_EINVAL;
    if (!valid_net(in_chns, C)) return UAPS_ERANGE;
    if (!aligned_to(params, 4) || !aligned_to(state, 16)) return UAPS_EALIGN;
    const Net n = make_net(in_chns, C);
    if (state_bytes < n.state_bytes) return UAPS_EINVAL;
    const size_t job_bytes = uaps_conv_pack_job_bytes();
    if (job_bytes > (size_t)kJobBytesMax || job_bytes % 4) return UAPS_EINVAL;
    unsigned char* st = static_cast<unsigned char*>(state);

    FoldArgs a{};
    a.params = params;
    a.state = st;
    UapsPackJob jobs[kLayers];
    long long total = 0;
    for (int i = 0; i < kLayers; ++i) {
        const Layer& L = n.l[i];
        FoldLayer& f = a.l[i];
        f.src = (long long)L.src; f.w_dst = (long long)L.w_off; f.b_dst = (long long)L.b_off;
        f.cout = L.cout; f.per_co = (L.cin1 + L.cin2) * L.ks * L.ks; f.bn = L.bn;
        f.first = total;
        total += (long long)L.cout * f.per_co + L.cout;
        jobs[i] = UapsPackJob{reinterpret_cast<const float*>(st + L.w_off), st + L.p_off, L.cout, L.cin1, L.cin2, L.ks, 0, 1};
    }
    a.total = total;
    std::vector<unsigned char> table(kLayers * job_bytes);
    int pack_blocks = 0;
    int rc = uaps_conv_pack_plan(jobs, kLayers, table.data(), &pack_blocks);
    if (rc != UAPS_OK) return rc;
    memcpy(a.table, table.data(), table.size());
    a.table_words = (int)(table.size() / 4);
    const long long blocks = ceil_div<long long>(total, 256);
    UAPS_LAUNCH(fold_bn_kernel, dim3((unsigned)(blocks < 1184 ? blocks : 1184)), dim3(256), 0, stream, a);
    UAPS_LAUNCH_CHECK();
    return uaps_conv_pack_run(st + n.table_off, kLayers, pack_blocks, stream);
}

UAPS_API int uaps_unet_infer_run(const void* state, size_t state_bytes, int in_chns, int C, const float* x, int B, int H,
                                 int W, void* workspace, size_t workspace_bytes, float* logits, uint8_t* labels,
                                 cudaStream_t stream) {
    if (state == nullptr || x == nullptr || workspace == nullptr || (logits == nullptr && labels == nullptr)) return UAPS_EINVAL;
    int rc = check_shape(B, H, W);
    if (rc != UAPS_OK) return rc;
    if (!valid_net(in_chns, C)) return UAPS_ERANGE;
    if (!aligned_to(state, 16) || !aligned_to(x, 16) || !aligned_to(workspace, 16) || (logits && !aligned_to(logits, 16)) ||
        (labels && !aligned_to(labels, 4)))
        return UAPS_EALIGN;
    const Net n = make_net(in_chns, C);
    const Ws w = ws_layout(B, H, W);
    if (state_bytes < n.state_bytes || workspace_bytes < w.bytes) return UAPS_EINVAL;

    const unsigned char* st = static_cast<const unsigned char*>(state);
    unsigned char* ws = static_cast<unsigned char*>(workspace);
    void* A = ws + w.a;
    void* Bf = ws + w.b;
    auto conv = [&](int i, const void* x1, const void* x2, void* out, int h, int wd, float slope, int nchw) {
        const Layer& L = n.l[i];
        const int c1s = i == 0 ? 16 : L.cin1;                         // the entry tensor holds pad16(in_chns) channels
        return uaps_conv_fprop_act(x1, c1s, x2, L.cin2, st + L.p_off, reinterpret_cast<const float*>(st + L.b_off), out,
                                   nchw ? 0 : L.cout, nchw, B, h, wd, L.cin1, L.cin2, L.cout, L.ks, nullptr, 0, 0, 1, slope,
                                   stream);
    };
    // encoder (UNet_UAPS._encode_folded)
    if ((rc = uaps_nchw_f32_to_nhwc_bf16(x, A, B, in_chns, H, W, 16, stream)) != UAPS_OK) return rc;
    for (int lvl = 0; lvl < 5; ++lvl) {
        const int h = H >> lvl, wd = W >> lvl;
        if (lvl && (rc = uaps_maxpool2_nhwc(ws + w.feat[lvl - 1], nullptr, A, B, 2 * h, 2 * wd, kFt[lvl - 1], stream)) != UAPS_OK)
            return rc;
        if ((rc = conv(2 * lvl, A, nullptr, Bf, h, wd, kSlope, 0)) != UAPS_OK) return rc;
        if ((rc = conv(2 * lvl + 1, Bf, nullptr, ws + w.feat[lvl], h, wd, kSlope, 0)) != UAPS_OK) return rc;
    }
    // main decoder (UNet_UAPS._decode_folded)
    const void* cur = ws + w.feat[4];
    for (int i = 1; i <= 4; ++i) {
        const int lvl = 4 - i, h = H >> lvl, wd = W >> lvl, k = 10 + 3 * (i - 1);
        if ((rc = conv(k, cur, nullptr, A, h / 2, wd / 2, 1.0f, 0)) != UAPS_OK) return rc;
        if ((rc = uaps_upsample2x_nhwc(A, Bf, B, h / 2, wd / 2, kFt[lvl], 0, stream)) != UAPS_OK) return rc;
        if ((rc = conv(k + 1, ws + w.feat[lvl], Bf, A, h, wd, kSlope, 0)) != UAPS_OK) return rc;
        if ((rc = conv(k + 2, A, nullptr, Bf, h, wd, kSlope, 0)) != UAPS_OK) return rc;
        cur = Bf;
    }
    float* z = logits != nullptr ? logits : reinterpret_cast<float*>(A);
    if ((rc = conv(kLayers - 1, cur, nullptr, z, H, W, 1.0f, 1)) != UAPS_OK) return rc;
    if (labels == nullptr) return UAPS_OK;
    switch (C) {
        case 2: return launch_labels<2>(z, labels, B, H * W, stream);
        case 3: return launch_labels<3>(z, labels, B, H * W, stream);
        case 4: return launch_labels<4>(z, labels, B, H * W, stream);
        case 5: return launch_labels<5>(z, labels, B, H * W, stream);
        case 6: return launch_labels<6>(z, labels, B, H * W, stream);
        case 7: return launch_labels<7>(z, labels, B, H * W, stream);
        case 8: return launch_labels<8>(z, labels, B, H * W, stream);
    }
    return UAPS_ERANGE;
}
