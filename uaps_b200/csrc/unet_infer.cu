// Whole-network inference through the C ABI, without PyTorch: the eval-mode forward of UNet_UAPS's encoder + main
// decoder (UAPS_unet.py:224-226, the output UAPS_train.py:377 and UAPS-Testing.ipynb keep), and the ensemble of every
// decoder with its perturbations and the uncertainty head (UAPS-Testing.ipynb cell 11).
//
// prepare folds every BatchNorm's running statistics into the convolution in front of it (one kernel, the arithmetic of
// UNet_UAPS._fold_bn) and packs all layers with one uaps_conv_pack_run launch.  uaps_unet_infer_run is UNet_UAPS.predict's
// folded forward -- the entry conversion, 23 conv launches with LeakyReLU in the epilogue, 4 max-pools, 4 upsamples,
// through the same entry points with the same arguments and in the same order -- plus an optional label map from the
// exact argmax of the softmax.  uaps_unet_ensemble_run is UNet_UAPS._ensemble_logits16 followed by
// ensemble.ensemble_uncertainty, launch for launch.  See include/uaps_b200.h for the contract, DESIGN.md f7 and f8.
#include <cstring>
#include <vector>

#include "argmax_exact.cuh"

namespace uaps {
namespace infer {

constexpr int kLayers = 23;                       // 5 encoder blocks x 2, 4 x (conv1x1 + 2), out_conv
constexpr int kDecLayers = 13;                    // one decoder: 4 x (conv1x1 + 2), out_conv
constexpr int kMaxAux = UAPS_KMAX - 1;            // auxiliary decoders of the ensemble entry points
constexpr int kMaxLayers = kLayers + kMaxAux * kDecLayers;
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
    Layer l[kMaxLayers];
    int n_layers;                  // kLayers + kDecLayers * n_aux
    size_t params;                 // floats in the blob
    size_t table_off;              // state offset of the pack-job table
    size_t state_bytes;
};

inline bool valid_net(int in_chns, int C) { return in_chns >= 1 && in_chns <= 16 && C >= 2 && C <= UAPS_CMAX; }
inline bool valid_aux(int n_aux) { return n_aux >= 1 && n_aux <= kMaxAux; }

// Layers in UNet_UAPS._main_plan order followed by n_aux auxiliary decoders in _aux_plan order, which is also state_dict
// order: per conv its weight and bias, then -- for the convs of a ConvBlock -- the BatchNorm's weight, bias, running_mean
// and running_var.  The state starts with the pack-job table; n_aux = 0 is the layout of uaps_unet_infer_*.
inline Net make_net(int in_chns, int C, int n_aux = 0) {
    Net n{};
    n.n_layers = kLayers + kDecLayers * n_aux;
    size_t src = 0, st = align_up((size_t)n.n_layers * kJobBytesMax);
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
    for (int d = 0; d <= n_aux; ++d) {                                // main_decoder, aux_decoder1..n_aux
        for (int i = 1; i <= 4; ++i) {                                // up1..4: conv1x1, conv (concat)
            const int c1 = kFt[5 - i], c2 = kFt[4 - i];
            add(c2, c1, 0, 1, 0);
            add(c2, c2, c2, 3, 1);
            add(c2, c2, 0, 3, 1);
        }
        add(C, kFt[0], 0, 3, 0);                                      // out_conv
    }
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
    FoldLayer l[kMaxLayers];
    long long total;
    int n_layers, table_words;
    uint32_t table[kMaxLayers * kJobBytesMax / 4];    // the host-built pack table, stored into the state by block 0
};
static_assert(sizeof(FoldArgs) <= 32764, "fold_bn_kernel's arguments must fit the kernel-parameter limit");

// w' = w * s, b' = (b - mean) * s + beta with s = gamma * rsqrt(var + eps): the ops and roundings of
// UNet_UAPS._fold_bn (torch's CUDA rsqrt is rsqrtf); layers without a BatchNorm are copied.
__global__ void __launch_bounds__(256) fold_bn_kernel(const __grid_constant__ FoldArgs a) {
    grid_dep_launch();
    grid_dep_wait();
    if (blockIdx.x == 0)
        for (int i = threadIdx.x; i < a.table_words; i += blockDim.x)
            reinterpret_cast<uint32_t*>(a.state)[i] = a.table[i];
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < a.total; e += (long long)gridDim.x * blockDim.x) {
        int lo = 0, hi = a.n_layers - 1;                              // last layer whose first element <= e
        while (lo < hi) {
            const int mid = (lo + hi + 1) >> 1;
            if (a.l[mid].first <= e) lo = mid; else hi = mid - 1;
        }
        const FoldLayer& f = a.l[lo];
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

inline size_t feat_bytes(int B, int H, int W, int lvl) { return (size_t)B * (H >> lvl) * (W >> lvl) * kFt[lvl] * 2; }

// workspace of uaps_unet_infer_run: the five encoder feature maps, then two scratch buffers of the largest activation
// (B*H*W*16 bf16 -- the entry tensor, every level-0 map; the fp32 logits when the caller passes none fit too, C <= 8)
struct Ws { size_t feat[5], a, b, bytes; };
inline Ws ws_layout(int B, int H, int W) {
    Ws w{};
    size_t off = 0;
    for (int l = 0; l < 5; ++l) {
        w.feat[l] = off;
        off = align_up(off + feat_bytes(B, H, W, l));
    }
    const size_t big = align_up((size_t)B * H * W * 16 * 2);
    w.a = off; w.b = off + big; w.bytes = off + 2 * big;
    return w;
}

// workspace of uaps_unet_ensemble_run: ws_layout's buffers, then the perturbed copies of the five feature maps for
// auxiliary decoders 1..min(n_aux, 3) (decoders 4 and 5 re-draw into the copies of decoders 1 and 2, which are decoded
// by then), FeatureDropout's attention map (one level at a time) and the five levels' smax words, the K logits, and the
// ensemble head's workspace
struct EnsWs { Ws base; size_t pert[3][5], att, smax, logits[UAPS_KMAX], head, head_bytes, bytes; };
inline EnsWs ens_ws_layout(int C, int n_aux, int B, int H, int W) {
    EnsWs w{};
    w.base = ws_layout(B, H, W);
    size_t off = w.base.bytes;
    for (int j = 0; j < n_aux && j < 3; ++j)
        for (int l = 0; l < 5; ++l) {
            w.pert[j][l] = off;
            off = align_up(off + feat_bytes(B, H, W, l));
        }
    w.att = off;
    w.smax = off;
    if (n_aux >= 3) {
        w.smax = off = align_up(off + (size_t)B * H * W * sizeof(float));
        off = align_up(off + 5 * (size_t)B * sizeof(uint32_t));
    }
    for (int k = 0; k <= n_aux; ++k) {
        w.logits[k] = off;
        off = align_up(off + (size_t)B * C * H * W * sizeof(float));
    }
    w.head = off;
    w.head_bytes = uaps_ensemble_workspace_bytes(1 + n_aux, C, B, (int64_t)H * W);
    w.bytes = align_up(off + w.head_bytes);
    return w;
}

inline int check_shape(int B, int H, int W) {
    if (B <= 0 || H <= 0 || W <= 0) return UAPS_EINVAL;
    if (H % 16 || W % 16) return UAPS_ERANGE;                          // four 2x poolings
    if (B > 65535 || (long long)B * H * W >= (1LL << 31)) return UAPS_ERANGE;
    return UAPS_OK;
}

// Perturbation launches of an ensemble forward (UNet_UAPS._ensemble_calls): one per level for auxiliary decoders 1-3
// together, then one per level for each of decoders 4 and 5.
inline int draws_count(int n_aux) { return 5 * (1 + (n_aux > 3 ? n_aux - 3 : 0)); }

constexpr float kNoiseRange = 0.3f;               // FeatureNoise(uniform_range=0.3) (UAPS_unet.py:172)
constexpr double kPDrop = 0.5;                    // Dropout(x, p=0.5) (:156)
constexpr float kUHost = 0.8f;                    // perturb3_nhwc's host u; the kernels read u from the draws

int prepare_net(const Net& n, const float* params, void* state, size_t state_bytes, cudaStream_t stream) {
    if (state_bytes < n.state_bytes) return UAPS_EINVAL;
    const size_t job_bytes = uaps_conv_pack_job_bytes();
    if (job_bytes > (size_t)kJobBytesMax || job_bytes % 4) return UAPS_EINVAL;
    unsigned char* st = static_cast<unsigned char*>(state);

    FoldArgs a{};
    a.params = params;
    a.state = st;
    a.n_layers = n.n_layers;
    UapsPackJob jobs[kMaxLayers];
    long long total = 0;
    for (int i = 0; i < n.n_layers; ++i) {
        const Layer& L = n.l[i];
        FoldLayer& f = a.l[i];
        f.src = (long long)L.src; f.w_dst = (long long)L.w_off; f.b_dst = (long long)L.b_off;
        f.cout = L.cout; f.per_co = (L.cin1 + L.cin2) * L.ks * L.ks; f.bn = L.bn;
        f.first = total;
        total += (long long)L.cout * f.per_co + L.cout;
        jobs[i] = UapsPackJob{reinterpret_cast<const float*>(st + L.w_off), st + L.p_off, L.cout, L.cin1, L.cin2, L.ks, 0, 1};
    }
    a.total = total;
    std::vector<unsigned char> table(n.n_layers * job_bytes);
    int pack_blocks = 0;
    int rc = uaps_conv_pack_plan(jobs, n.n_layers, table.data(), &pack_blocks);
    if (rc != UAPS_OK) return rc;
    memcpy(a.table, table.data(), table.size());
    a.table_words = (int)(table.size() / 4);
    const long long blocks = ceil_div<long long>(total, 256);
    UAPS_LAUNCH(fold_bn_kernel, dim3((unsigned)(blocks < 1184 ? blocks : 1184)), dim3(256), 0, stream, a);
    UAPS_LAUNCH_CHECK();
    return uaps_conv_pack_run(st + n.table_off, n.n_layers, pack_blocks, stream);
}

int layer_offsets(const Net& n, int layer, size_t* weight_offset, size_t* bias_offset, size_t* packed_offset,
                  size_t* packed_bytes) {
    if (layer < 0 || layer >= n.n_layers) return UAPS_ERANGE;
    const Layer& L = n.l[layer];
    *weight_offset = L.w_off; *bias_offset = L.b_off; *packed_offset = L.p_off; *packed_bytes = L.p_bytes;
    return UAPS_OK;
}

// The folded forward's two walks over a prepared state, shared by both run entry points; a and b are ws_layout's two
// scratch buffers.
struct Forward {
    const Net& n;
    const unsigned char* st;
    void* a;
    void* b;
    int B, H, W;
    cudaStream_t stream;

    int conv(int i, const void* x1, const void* x2, void* out, int h, int wd, float slope, int nchw) const {
        const Layer& L = n.l[i];
        const int c1s = i == 0 ? 16 : L.cin1;                         // the entry tensor holds pad16(in_chns) channels
        return uaps_conv_fprop_act(x1, c1s, x2, L.cin2, st + L.p_off, reinterpret_cast<const float*>(st + L.b_off), out,
                                   nchw ? 0 : L.cout, nchw, B, h, wd, L.cin1, L.cin2, L.cout, L.ks, nullptr, 0, 0, 1, slope,
                                   stream);
    }

    // UNet_UAPS._encode_folded: x [B, in_chns, H, W] fp32 -> feat[l] = level l's map [B, H_l, W_l, C_l] bf16
    int encode(const float* x, int in_chns, void* const* feat) const {
        int rc = uaps_nchw_f32_to_nhwc_bf16(x, a, B, in_chns, H, W, 16, stream);
        if (rc != UAPS_OK) return rc;
        for (int lvl = 0; lvl < 5; ++lvl) {
            const int h = H >> lvl, wd = W >> lvl;
            if (lvl && (rc = uaps_maxpool2_nhwc(feat[lvl - 1], nullptr, a, B, 2 * h, 2 * wd, kFt[lvl - 1], stream)) != UAPS_OK)
                return rc;
            if ((rc = conv(2 * lvl, a, nullptr, b, h, wd, kSlope, 0)) != UAPS_OK) return rc;
            if ((rc = conv(2 * lvl + 1, b, nullptr, feat[lvl], h, wd, kSlope, 0)) != UAPS_OK) return rc;
        }
        return UAPS_OK;
    }

    // UNet_UAPS._decode_folded: the decoder whose up1.conv1x1 is layer `first`, over feat -> z [B, C, H, W] fp32
    int decode(const void* const* feat, int first, float* z) const {
        int rc;
        const void* cur = feat[4];
        for (int i = 1; i <= 4; ++i) {
            const int lvl = 4 - i, h = H >> lvl, wd = W >> lvl, k = first + 3 * (i - 1);
            if ((rc = conv(k, cur, nullptr, a, h / 2, wd / 2, 1.0f, 0)) != UAPS_OK) return rc;
            if ((rc = uaps_upsample2x_nhwc(a, b, B, h / 2, wd / 2, kFt[lvl], 0, stream)) != UAPS_OK) return rc;
            if ((rc = conv(k + 1, feat[lvl], b, a, h, wd, kSlope, 0)) != UAPS_OK) return rc;
            if ((rc = conv(k + 2, a, nullptr, b, h, wd, kSlope, 0)) != UAPS_OK) return rc;
            cur = b;
        }
        return conv(first + kDecLayers - 1, cur, nullptr, z, H, W, 1.0f, 1);
    }
};

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
    if (!valid_net(in_chns, C)) return UAPS_ERANGE;
    return layer_offsets(make_net(in_chns, C), layer, weight_offset, bias_offset, packed_offset, packed_bytes);
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
    return prepare_net(make_net(in_chns, C), params, state, state_bytes, stream);
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

    unsigned char* ws = static_cast<unsigned char*>(workspace);
    const Forward f{n, static_cast<const unsigned char*>(state), ws + w.a, ws + w.b, B, H, W, stream};
    void* feat[5];
    for (int l = 0; l < 5; ++l) feat[l] = ws + w.feat[l];
    if ((rc = f.encode(x, in_chns, feat)) != UAPS_OK) return rc;
    float* z = logits != nullptr ? logits : reinterpret_cast<float*>(ws + w.a);
    if ((rc = f.decode(feat, kLayers - kDecLayers, z)) != UAPS_OK) return rc;
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

// ---- ensemble: every decoder, its perturbations and the uncertainty head ---------------------------------------------
UAPS_API size_t uaps_unet_ensemble_params_count(int in_chns, int C, int n_aux) {
    return valid_net(in_chns, C) && valid_aux(n_aux) ? make_net(in_chns, C, n_aux).params : 0;
}

UAPS_API size_t uaps_unet_ensemble_state_bytes(int in_chns, int C, int n_aux) {
    return valid_net(in_chns, C) && valid_aux(n_aux) ? make_net(in_chns, C, n_aux).state_bytes : 0;
}

UAPS_API size_t uaps_unet_ensemble_draws_count(int n_aux) { return valid_aux(n_aux) ? (size_t)draws_count(n_aux) : 0; }

UAPS_API size_t uaps_unet_ensemble_workspace_bytes(int in_chns, int C, int n_aux, int B, int H, int W) {
    if (!valid_net(in_chns, C) || !valid_aux(n_aux) || check_shape(B, H, W) != UAPS_OK) return 0;
    return ens_ws_layout(C, n_aux, B, H, W).bytes;
}

UAPS_API int uaps_unet_ensemble_layer(int in_chns, int C, int n_aux, int layer, size_t* weight_offset, size_t* bias_offset,
                                      size_t* packed_offset, size_t* packed_bytes) {
    if (weight_offset == nullptr || bias_offset == nullptr || packed_offset == nullptr || packed_bytes == nullptr) return UAPS_EINVAL;
    if (!valid_net(in_chns, C) || !valid_aux(n_aux)) return UAPS_ERANGE;
    return layer_offsets(make_net(in_chns, C, n_aux), layer, weight_offset, bias_offset, packed_offset, packed_bytes);
}

UAPS_API int uaps_unet_ensemble_prepare(const float* params, int in_chns, int C, int n_aux, void* state, size_t state_bytes,
                                        cudaStream_t stream) {
    if (params == nullptr || state == nullptr) return UAPS_EINVAL;
    if (!valid_net(in_chns, C) || !valid_aux(n_aux)) return UAPS_ERANGE;
    if (!aligned_to(params, 4) || !aligned_to(state, 16)) return UAPS_EALIGN;
    return prepare_net(make_net(in_chns, C, n_aux), params, state, state_bytes, stream);
}

UAPS_API int uaps_unet_ensemble_run(const void* state, size_t state_bytes, int in_chns, int C, int n_aux, const float* x,
                                    int B, int H, int W, const int64_t* draws, void* workspace, size_t workspace_bytes,
                                    uint8_t* labels, float* uncertainty, float* image_uncertainty, float* mean_prob,
                                    cudaStream_t stream) {
    if (state == nullptr || x == nullptr || draws == nullptr || workspace == nullptr || labels == nullptr) return UAPS_EINVAL;
    int rc = check_shape(B, H, W);
    if (rc != UAPS_OK) return rc;
    if (!valid_net(in_chns, C) || !valid_aux(n_aux)) return UAPS_ERANGE;
    // 16-byte outputs make uaps_ensemble_head take the vector width it takes for torch's allocations; its per-image
    // fp64 fold is chunked by that width, so this is what keeps image_uncertainty bit-equal to the Python path
    if (!aligned_to(state, 16) || !aligned_to(x, 16) || !aligned_to(draws, 8) || !aligned_to(workspace, 16) ||
        !aligned_to(labels, 4) || !aligned_to(uncertainty, 16) || !aligned_to(image_uncertainty, 16) ||
        !aligned_to(mean_prob, 16))
        return UAPS_EALIGN;
    const Net n = make_net(in_chns, C, n_aux);
    const EnsWs w = ens_ws_layout(C, n_aux, B, H, W);
    if (state_bytes < n.state_bytes || workspace_bytes < w.bytes) return UAPS_EINVAL;

    unsigned char* ws = static_cast<unsigned char*>(workspace);
    const Forward f{n, static_cast<const unsigned char*>(state), ws + w.base.a, ws + w.base.b, B, H, W, stream};
    void* feat[5];
    for (int l = 0; l < 5; ++l) feat[l] = ws + w.base.feat[l];
    if ((rc = f.encode(x, in_chns, feat)) != UAPS_OK) return rc;

    // draws: int64 [2][n_calls]; column i = Philox key (row 0) and FeatureDropout u (row 1, fp32 in the low 4 bytes) of
    // perturbation launch i, read by the kernels only
    const int n_calls = draws_count(n_aux);
    const uint64_t* keys = reinterpret_cast<const uint64_t*>(draws);
    float* att = reinterpret_cast<float*>(ws + w.att);
    uint32_t* smax = reinterpret_cast<uint32_t*>(ws + w.smax);
    auto perturb = [&](int call, int lvl, void* y_noise, void* y_drop, void* y_fdrop) {
        const int64_t hw = (int64_t)(H >> lvl) * (W >> lvl);
        uint32_t* sm = y_fdrop != nullptr ? smax + (size_t)lvl * B : nullptr;
        int r;
        if (y_fdrop != nullptr && (r = uaps_fdrop_stats_nhwc(feat[lvl], B, kFt[lvl], hw, att, sm, stream)) != UAPS_OK) return r;
        return uaps_perturb3_nhwc(feat[lvl], 0, kNoiseRange, kPDrop, y_fdrop != nullptr ? att : nullptr, sm, kUHost, y_noise,
                                  y_drop, y_fdrop, B, kFt[lvl], hw, keys + call,
                                  reinterpret_cast<const float*>(draws + n_calls + call), stream);
    };
    if (n_aux >= 3) {                                                  // FeatureDropout's smax words, all five levels
        const cudaError_t e = cudaMemsetAsync(smax, 0, 5 * (size_t)B * sizeof(uint32_t), stream);
        if (e != cudaSuccess) return (int)e;
    }
    for (int lvl = 0; lvl < 5; ++lvl) {                                // one launch per level for decoders 1..min(n_aux, 3)
        void* y[3] = {nullptr, nullptr, nullptr};
        for (int j = 0; j < n_aux && j < 3; ++j) y[j] = ws + w.pert[j][lvl];
        if ((rc = perturb(lvl, lvl, y[0], y[1], y[2])) != UAPS_OK) return rc;
    }
    float* z[UAPS_KMAX];
    for (int k = 0; k <= n_aux; ++k) z[k] = reinterpret_cast<float*>(ws + w.logits[k]);
    if ((rc = f.decode(feat, kLayers - kDecLayers, z[0])) != UAPS_OK) return rc;
    for (int a = 1; a <= n_aux; ++a) {
        const int j = (a - 1) % 3;                                     // family: noise, dropout, feature dropout
        void* pf[5];
        for (int l = 0; l < 5; ++l) pf[l] = ws + w.pert[j][l];
        for (int lvl = 0; a > 3 && lvl < 5; ++lvl) {                   // decoders 4, 5: a fresh draw of their family
            void* y[3] = {nullptr, nullptr, nullptr};
            y[j] = pf[lvl];
            if ((rc = perturb(5 * (a - 3) + lvl, lvl, y[0], y[1], y[2])) != UAPS_OK) return rc;
        }
        if ((rc = f.decode(pf, kLayers + kDecLayers * (a - 1), z[a])) != UAPS_OK) return rc;
    }
    return uaps_ensemble_head(z, 1 + n_aux, B, C, (int64_t)H * W, labels, uncertainty, image_uncertainty, mean_prob,
                              ws + w.head, w.head_bytes, stream);
}
