/*
 * uaps_b200.h -- C ABI of libuaps_b200.so: the UAPS unlabeled-batch hot path on B200 (sm_100a).
 *
 * The reference (djene-mengistu/UAPS) has no FFI: its hot path is Python over torch.nn.  This
 * header is the boundary a maintainer binds *underneath* that Python surface (ctypes stub in
 * INTEGRATION.md).  Each entry point names the reference expression it replaces, with
 * file:line relative to the reference checkout.
 *
 * Conventions (all entry points)
 *   - plain pointers and sizes; every buffer is allocated and owned by the CALLER; the library
 *     never allocates device memory, never retains a pointer past the call, never synchronises
 *     the host, and launches only on the stream it is given (re-entrant per device/stream);
 *   - tensors are contiguous NCHW fp32 unless stated otherwise, exactly as the reference's
 *     model emits them (utilities/UAPS_unet.py:224-233);
 *   - return value: 0 = ok, negative = UAPS_E* (invalid argument), positive = cudaError_t of
 *     the failed launch.  Nothing throws across the ABI.
 */
#ifndef UAPS_B200_H
#define UAPS_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#ifndef __DRIVER_TYPES_H__
typedef struct CUstream_st* cudaStream_t;
#endif

#define UAPS_ABI_VERSION 2
#define UAPS_KMAX 6              /* decoders: reference uses 4 (UAPS_unet.py:219-222); ablation up to 5 */
#define UAPS_CMAX 8              /* classes: 4 NEU, 2 KoSDD2, 7 DAGM (DAGM-Dataset-codes/UAPS_model.py:11) */

enum {
    UAPS_OK = 0,
    UAPS_EINVAL = -1,            /* null pointer, non-positive size */
    UAPS_ERANGE = -2,            /* K, C or pixel count outside the supported range */
    UAPS_EALIGN = -3,            /* pointer not aligned to its element type */
    UAPS_ENODEV = -4             /* not running on an sm_100 device */
};

int         uaps_abi_version(void);
const char* uaps_error_string(int code);

/* ---------------------------------------------------------------------------------------------
 * Device-resident per-iteration state.  The reference's loop draws its per-iteration scalars on the HOST
 * (np.random.dirichlet :251, np.random.uniform UAPS_unet.py:165, the ramp :279-280, Adam's step count) and
 * passes them to kernels by value; that forces ~1150 launches per iteration through Python.  Here they live in
 * one small device struct advanced by ONE single-thread kernel (uaps_step_begin) at the top of the iteration,
 * and every entry point below that used to take such a scalar also takes a nullable device pointer into this
 * struct, so a whole iteration (two forwards, both losses, backward, optimizer) is a static launch sequence
 * that can be captured once into a CUDA graph and replayed.
 * ------------------------------------------------------------------------------------------- */
#define UAPS_STEP_USLOTS 16
typedef struct UapsStepState {
    uint64_t iter;              /* completed iterations; the ramp "epoch" is iter / iters_per_ramp_epoch (:279-280) */
    uint64_t key_rank;          /* Philox key offset of this iteration for per-rank draws (dropout masks, feature noise) */
    uint64_t key_shared;        /* the same for draws every rank must agree on                                       */
    uint64_t adam_step;         /* optimizer steps taken (bias correction)                                            */
    uint32_t xchg_base;         /* exchange epochs of this iteration are xchg_base + 1 .. xchg_base + n_exchanges      */
    uint32_t xchg_next;
    uint32_t skipped;           /* written by uaps_adam_step: 1 = the loss was not finite, the update was skipped      */
    uint32_t n_skipped;         /* how often that happened (latched, never reset by the library)                       */
    float lr;                   /* HOST-written learning rate (a scheduler edits it, :113); read by uaps_step_begin     */
    float adam_step_size;       /* lr / (1 - beta1^t)                                                                  */
    float adam_inv_bc2_sqrt;    /* 1 / sqrt(1 - beta2^t)                                                               */
    float reserved;
    float mix_w[8];             /* Dirichlet(1,...,1) draw over the K decoders (:251), fp32-rounded                    */
    float cw1, cw2;             /* consistency_i * sigmoid_rampup(iter / iters_per_ramp_epoch, rampup_length)          */
    float u[UAPS_STEP_USLOTS];  /* FeatureDropout thresholds U(0.7, 0.9) (UAPS_unet.py:165), one per call of the step  */
} UapsStepState;
/* float offsets inside the `wcw` block (&state->mix_w[0]) the loss entry points take */
#define UAPS_WCW_CW1 8
#define UAPS_WCW_CW2 9

/* Advance `state` (device, zero-initialised once, 16-byte aligned) by one iteration: draws mix_w (K weights), the
 * n_u thresholds and the two Philox keys from Philox4x32-10 keyed by (seed_shared | seed_rank, iter), evaluates the
 * ramp in fp64 (utilities/ramps.py:19-26), Adam's bias corrections for step adam_step + 1 (not advanced when the
 * previous update was skipped), moves the exchange-epoch window by n_exchanges, and increments iter. */
int uaps_step_begin(UapsStepState* state, uint64_t seed_rank, uint64_t seed_shared, int K, int n_u,
                    double consistency1, double consistency2, double rampup_length, int iters_per_ramp_epoch,
                    int n_exchanges, float beta1, float beta2, cudaStream_t stream);

/* ---------------------------------------------------------------------------------------------
 * Fused pseudo-label + KL-uncertainty + uncertainty-weighted CE/Dice loss
 * replaces UAPS_train.py:186-189 (K softmaxes), :223 (mean prediction), :226-236 (KL maps and
 * exp(-KL)), :241-243 (uncertainty loss), :251-255 (Dirichlet mix + argmax), :259-262 with
 * utilities/pytorch_losses.py:54-89 (CE + Dice per decoder), :265-277 (uncertainty weighting),
 * :282 (unlabeled part of the total) and their autograd backward (:287).
 *
 * Two passes are forced by the math: every per-pixel gradient needs batch-global scalars.
 *   pass1    : read K logits tensors once, per-pixel softmax/KL/argmax in registers, warp-shuffle
 *              + block partial sums, last block folds them to `sums` in fp64 (deterministic).
 *   (N>1 GPUs: the caller all-reduces `sums` here -- the path's one data exchange.)
 *   finalize : sums -> loss scalars.
 *   pass2    : re-read logits, recompute per-pixel terms, write d(loss)/d(logits).
 * Algorithmic HBM bytes per unlabeled pixel: pass1 4KC, pass2 8KC (read 4KC + write 4KC).
 * ------------------------------------------------------------------------------------------- */

/* number of doubles in `sums`: [K] sum(-logp[y]) | [K] sum(E_k) | [K] sum(V_k) | [K*C] I_kc |
 * [K*C] sum(p_kc) | [C] T_c = count(y == c). */
int    uaps_loss_sums_count(int K, int C);
/* number of floats in `scalars` (layout: UAPS_SC_* below). */
int    uaps_loss_scalars_count(int K, int C);
/* bytes of scratch `workspace` pass1 needs.  Must be zero-filled ONCE by the caller before its
 * first use; every call leaves it ready for the next one. */
size_t uaps_loss_workspace_bytes(int K, int C);

/* scalars[] layout */
#define UAPS_SC_LOSS_U   0       /* cw1 * ps_loss + cw2 * l_uncert      (UAPS_train.py:282)      */
#define UAPS_SC_PS_LOSS  1       /* (1/K) sum_k ps_k * mean(E_k)        (:265-277)               */
#define UAPS_SC_L_UNCERT 2       /* mean((1/K) sum_k V_k)               (:241-243)               */
#define UAPS_SC_CW1      3
#define UAPS_SC_CW2      4
#define UAPS_SC_INV_N    5       /* 1 / N_global                                                   */
#define UAPS_SC_MEAN_CE  6       /* mean_k CE_k    (total_loss_ce,   UAPS_train.py:216)            */
#define UAPS_SC_MEAN_DICE 7      /* mean_k Dice_k  (total_loss_dice, UAPS_train.py:217)            */
#define UAPS_SC_BASE     8       /* then ps_k[K], Ebar_k[K], CE_k[K], Dice_k[K], I_kc[K*C], Card_kc[K*C] */

/* flags for pass1 / pass2 (must be the same in both).
 * default (0): MUFU-based exp2/log2/rcp arithmetic, values within ~1e-6 relative of the fp32
 *   reference; the pseudo-label is STILL bit-exact with torch.argmax: pixels whose top-two mixed
 *   probabilities are closer than 2e-5 are re-decided with the exact torch-order chain.
 * UAPS_LOSS_EXACT: every softmax uses torch's op order and IEEE expf/div/logf (validation mode,
 *   about half the speed). */
#define UAPS_LOSS_EXACT 1

/* z: host array of K device pointers, each [B,C,HW] fp32.  mix_w: host array of K floats (the
 * Dirichlet draw of :251, already rounded to fp32 as torch rounds a python scalar).
 * labels: NULL for the unlabeled path (pseudo-label = argmax of the mix); else device int64
 * [B,HW] ground truth -> supervised mode (UAPS_train.py:194-218: no KL terms, E_k = 1).
 * pseudo_out: nullable device int64 [B,HW] (torch.argmax result, lowest index on ties).
 * exp_var_out: nullable host array of K device pointers [B,HW] fp32 receiving exp(-V_k). */
int uaps_loss_pass1(const float* const* z, int K, int B, int C, int64_t HW,
                    const float* mix_w, const int64_t* labels,
                    void* workspace, double* sums,
                    int64_t* pseudo_out, float* const* exp_var_out, int flags, cudaStream_t stream);

/* Single-rank fast path: pass 1 followed by ONE kernel that folds the partial sums and writes the scalars
 * (N_global = B * HW), i.e. uaps_loss_pass1 + uaps_loss_finalize with a launch less.  `sums` is still written. */
int uaps_loss_pass1_scalars(const float* const* z, int K, int B, int C, int64_t HW,
                            const float* mix_w, const int64_t* labels, void* workspace, double* sums,
                            int64_t* pseudo_out, float* const* exp_var_out, int flags,
                            float cw1, float cw2, float* scalars,
                            const float* wcw_dev, /* nullable: &UapsStepState.mix_w[0]; then mix_w / cw1 / cw2 are read from the device */
                            cudaStream_t stream);

/* ---- multi-GPU exchange (replaces the DataParallel gather of UAPS_model.py:13 for the loss sums) ----------
 * One process per GPU, all on one NVLink/NVSwitch domain.  Each rank owns a MAILBOX (device memory allocated by
 * uaps_xchg_alloc -- the one allocation this library makes, because CUDA IPC needs the allocation base) and maps
 * every peer's mailbox through a 64-byte handle exchanged out of band (torch.distributed in uaps_b200/comm.py).
 * uaps_loss_pass1_exchange = pass 1, then ONE kernel that folds the partial sums, stores them into every rank's
 * mailbox over NVLink (8-byte words carrying 32 data bits + the epoch tag, so data and flag arrive together), collects
 * the world's words from its own mailbox and finalizes the scalars -- no NCCL call on the data path.
 * mailboxes: host array of `world` device pointers as mapped in THIS process (own mailbox at [rank]);
 * epoch: 1, 2, 3, ... incremented by the caller per exchange, identical on all ranks; N_global: pixels of the
 * whole batch.  A peer that never arrives (UAPS_XCHG_TIMEOUT_MS, default 4000) turns the scalars into NaN and
 * latches the epoch into the status word (uaps_xchg_status) instead of hanging the GPU. */
#define UAPS_XCHG_MAX_RANKS 8
size_t uaps_xchg_mailbox_bytes(void);
int uaps_xchg_alloc(void** mailbox);
int uaps_xchg_free(void* mailbox);
int uaps_xchg_export(void* mailbox, void* handle64);
int uaps_xchg_import(const void* handle64, void** peer_mailbox);
int uaps_xchg_close(void* peer_mailbox);
int uaps_xchg_status(const void* mailbox, unsigned* status_out, cudaStream_t stream);
int uaps_loss_pass1_exchange(const float* const* z, int K, int B, int C, int64_t HW,
                             const float* mix_w, const int64_t* labels, void* workspace, double* sums,
                             int64_t* pseudo_out, float* const* exp_var_out, int flags,
                             void* const* mailboxes, int rank, int world, unsigned epoch, int64_t N_global,
                             float cw1, float cw2, float* scalars,
                             const float* wcw_dev,        /* nullable, as above */
                             const uint32_t* epoch_dev,   /* nullable: &UapsStepState.xchg_base; the epoch used is *epoch_dev + epoch */
                             cudaStream_t stream);

/* sums_global: device, uaps_loss_sums_count doubles (all-reduced over ranks by the caller when
 * the batch is sharded); N_global = total pixels behind those sums.  supervised != 0 selects
 * the labeled-batch formula (scalars[LOSS_U] = mean_k 0.5(CE_k + Dice_k), cw ignored). */
int uaps_loss_finalize(const double* sums_global, int K, int C, int64_t N_global,
                       float cw1, float cw2, int supervised, float* scalars, cudaStream_t stream);

/* grad_out: device, laid out like scalars[]: the upstream gradients of the five differentiable
 * slots LOSS_U, PS_LOSS, L_UNCERT, MEAN_CE, MEAN_DICE are read, the rest ignored (so the autograd
 * gradient of the scalars vector can be passed as is).
 * dz: host array of K device pointers [B,C,HW] fp32, overwritten. */
int uaps_loss_pass2(const float* const* z, int K, int B, int C, int64_t HW,
                    const float* mix_w, const int64_t* labels,
                    const float* scalars, const float* grad_out,
                    float* const* dz, int flags, const float* wcw_dev /* nullable, as in pass 1 */, cudaStream_t stream);

/* ---------------------------------------------------------------------------------------------
 * Ensemble inference head: the test-time uncertainty of the K decoders (UAPS-Testing.ipynb cell 11) from the
 * expressions of the uncertainty loss, per pixel, with no loss sums:
 *   labels[b,hw]            = argmax_c q (uint8, lowest index on ties), q = (((p_0 + p_1) + ...) / K) and
 *                             p_k = softmax(z_k) (UAPS_train.py:186-189, 223) -- bit-exact with torch.argmax(q, 1)
 *                             by the same near-tie rule as the pseudo-label of pass 1;
 *   uncertainty[b,hw]       = (1/K) sum_k V_k, V_k = sum_c KLDiv(log_softmax(z_k), q) (:226-236), the per-pixel
 *                             term of the uncertainty loss (:241-243);
 *   image_uncertainty[b]    = mean of uncertainty over the HW pixels of image b, summed in fp64 in a fixed order
 *                             (bitwise reproducible);
 *   mean_prob[b,c,hw]       = q.
 * z: host array of K device pointers [B,C,HW] fp32 (1 <= K <= UAPS_KMAX, 2 <= C <= UAPS_CMAX, any HW).
 * uncertainty, image_uncertainty and mean_prob are nullable.  image_uncertainty needs a workspace of at least
 * uaps_ensemble_workspace_bytes(K, C, B, HW) bytes, 8-byte aligned; every launch writes the part it reads, so it
 * needs no initialisation and the call can be captured into a CUDA graph and replayed.
 * Algorithmic HBM bytes per pixel: 4KC read + 1 (label) + 4 (uncertainty) written, + 4C with mean_prob.
 * ------------------------------------------------------------------------------------------- */
size_t uaps_ensemble_workspace_bytes(int K, int C, int B, int64_t HW);
int uaps_ensemble_head(const float* const* z, int K, int B, int C, int64_t HW, uint8_t* labels, float* uncertainty,
                       float* image_uncertainty, float* mean_prob, void* workspace, size_t workspace_bytes,
                       cudaStream_t stream);

/* ---------------------------------------------------------------------------------------------
 * Encoder-feature perturbations (utilities/UAPS_unet.py:156-185, applied at :227-231).
 * x, y: [B, C, HW] fp32 (C*HW = `chw` elements per sample where only that matters).
 * Randomness is either INJECTED (a caller-provided tensor, used for parity with the reference's
 * draws) or generated in-kernel from a Philox4x32-10 counter keyed by (seed, element index), so
 * forward and backward regenerate the same draw and no mask is ever stored.
 * ------------------------------------------------------------------------------------------- */

/* FeatureNoise :172-185: y = x * n + x, n ~ U(-range, range) of shape [C,HW], shared by the batch.
 * noise == NULL -> Philox(seed).  The same entry point is its backward (dx = g * n + g). */
int uaps_feature_noise(const float* x, const float* noise, uint64_t seed, float range,
                       float* y, int B, int64_t chw, cudaStream_t stream);

/* F.dropout(x, p) with training=True (:156-158) and nn.Dropout(p) of the encoder blocks (:40):
 * y = x * keep / (1 - p).  keep (uint8 [B*chw]) == NULL -> Philox(seed).  Also its own backward. */
int uaps_dropout(const float* x, const uint8_t* keep, uint64_t seed, double p,
                 float* y, int64_t n, cudaStream_t stream);

/* FeatureDropout :161-169, phase 1: attention[b,hw] = mean_c x[b,c,hw]; smax[b] = max_hw attention.
 * smax_enc (B uint32, order-preserving encoding of the float max) must be zeroed by the caller. */
int uaps_fdrop_stats(const float* x, int B, int C, int64_t HW,
                     float* attention, uint32_t* smax_enc, cudaStream_t stream);
/* phase 2: y = x * (attention < smax * u), u = the single U(0.7,0.9) draw of :165 (host float).
 * With x := upstream gradient it is the backward (the comparison carries no gradient). */
int uaps_fdrop_apply(const float* x, const float* attention, const uint32_t* smax_enc, float u,
                     float* y, int B, int C, int64_t HW, cudaStream_t stream);

/* All three at once for one feature level: x is read once, three perturbed copies are written
 * (16 B/element instead of 24).  Any of y_noise / y_drop / y_fdrop may be NULL. */
int uaps_perturb3(const float* x, const float* noise, const uint8_t* keep, uint64_t seed,
                  float noise_range, double p_drop, const float* attention,
                  const uint32_t* smax_enc, float u,
                  float* y_noise, float* y_drop, float* y_fdrop,
                  int B, int C, int64_t HW, cudaStream_t stream);

/* Backward of uaps_perturb3: dx = g_noise*n + g_noise + g_drop*keep/(1-p) + g_fdrop*mask, one pass.
 * Any of the three upstream gradients may be NULL (that branch had no consumer). */
int uaps_perturb3_bwd(const float* g_noise, const float* g_drop, const float* g_fdrop,
                      const float* noise, const uint8_t* keep, uint64_t seed, float noise_range,
                      double p_drop, const float* attention, const uint32_t* smax_enc, float u,
                      float* dx, int B, int C, int64_t HW, cudaStream_t stream);

/* Channels-last bf16 versions of the perturbations for the bf16 / tcgen05 model path: x is
 * [B, HW, C] bf16, C in {8, 16, ..., 256} (power of two), HW * C / 8 a multiple of 32.  Philox only.
 * Same three outputs as uaps_perturb3 (any may be NULL); the _bwd entry folds the three upstream
 * gradients into dx through the regenerated masks. */
int uaps_fdrop_stats_nhwc(const void* x, int B, int C, int64_t HW, float* attention,
                          uint32_t* smax_enc, cudaStream_t stream);
int uaps_perturb3_nhwc(const void* x, uint64_t seed, float noise_range, double p_drop,
                       const float* attention, const uint32_t* smax_enc, float u,
                       void* y_noise, void* y_drop, void* y_fdrop, int B, int C, int64_t HW,
                       const uint64_t* seed_dev, /* nullable: *seed_dev is added to seed (&UapsStepState.key_rank) */
                       const float* u_dev,       /* nullable: overrides u (&UapsStepState.u[slot]) */
                       cudaStream_t stream);
int uaps_perturb3_nhwc_bwd(const void* g_noise, const void* g_drop, const void* g_fdrop, uint64_t seed,
                           float noise_range, double p_drop, const float* attention,
                           const uint32_t* smax_enc, float u, void* dx, int B, int C, int64_t HW,
                           const uint64_t* seed_dev, const float* u_dev,
                           const void* g_extra1, const void* g_extra2, /* nullable: gradients of UNPERTURBED uses of x (the main
                              decoder's skip connection, the next level's max-pool), added to dx in the same pass */
                           cudaStream_t stream);

/* nn.Upsample(scale_factor=2, mode='bilinear', align_corners=True) (utilities/UAPS_unet.py:74-75) and
 * nn.MaxPool2d(2) (:56) on channels-last bf16, C % 8 == 0.
 * upsample: backward = 0: x [B,H,W,C] -> y [B,2H,2W,C]; backward = 1: x is the upstream gradient
 *   [B,2H,2W,C] and y receives d input [B,H,W,C] (gather form, deterministic).  H, W = INPUT size.
 * maxpool: gy == NULL: out [B,H/2,W/2,C] = max of 2x2 windows of x [B,H,W,C]; gy given: out = d x, the
 *   gradient routed to the first maximum of each window (torch's tie rule). */
int uaps_upsample2x_nhwc(const void* x, void* y, int B, int H, int W, int C, int backward, cudaStream_t stream);
int uaps_maxpool2_nhwc(const void* x, const void* gy, void* out, int B, int H, int W, int C, cudaStream_t stream);

/* [B,C,H,W] fp32 NCHW -> [B,H,W,Cp] bf16 channels-last, channels C..Cp-1 zero-filled (Cp % 8 == 0, Cp >= C): the
 * entry into the bf16 path for the network input (UAPS_train.py:177,185 feed NCHW fp32 batches) and for the
 * fp32 logits gradient coming back from the fused loss. */
int uaps_nchw_f32_to_nhwc_bf16(const float* x, void* out, int B, int C, int H, int W, int Cp, cudaStream_t stream);
/* The same for C <= 8 (the logits gradient), also accumulating the per-channel sums over all pixels of the bf16 values it
 * writes -- the bias gradient of out_conv (utilities/UAPS_unet.py:138-139, through loss.backward() at UAPS_train.py:287):
 * sums = uaps_nchw_f32_to_nhwc_bf16_sums_nrep() replicas of [Cp] doubles, zeroed by the caller; the total is their sum. */
int uaps_nchw_f32_to_nhwc_bf16_sums_nrep(void);
int uaps_nchw_f32_to_nhwc_bf16_sums(const float* x, void* out, int B, int C, int H, int W, int Cp, double* sums,
                                    cudaStream_t stream);

/* Fused train-mode BatchNorm2d + LeakyReLU(slope) + Dropout(p) on channels-last bf16 activations
 * (utilities/UAPS_unet.py:37-43: nn.BatchNorm2d -> nn.LeakyReLU() -> nn.Dropout(p)).  y: [npix, C] bf16,
 * C a power of two in 8..256.  sum / sumsq: device fp64 [C], zeroed by the caller before _stats.
 * _act normalises with the batch statistics, writes save_mean / save_rstd [C] and (if given) advances
 * running_mean / running_var with `momentum` (unbiased variance), as torch does.  The backward entry
 * recomputes the LeakyReLU sign and the Philox dropout mask from y and the seed; sum_g / sum_gx (fp64 [C],
 * zeroed by the caller) return sum(g') = d(beta) and the RAW second moment sum(g' * y), from which
 * d(gamma) = save_rstd * (sum_gx - save_mean * sum_g) (the dgamma_accum / dbeta_accum path applies that itself). */
int uaps_bn_stats_nhwc(const void* y, int64_t npix, int C, double* sum, double* sumsq, cudaStream_t stream);
int uaps_bn_act_nhwc(const void* y, const double* sum, const double* sumsq, const float* gamma,
                     const float* beta, float* running_mean, float* running_var, float momentum,
                     float eps, float slope, double p_drop, uint64_t seed, void* out,
                     float* save_mean, float* save_rstd, int64_t npix, int C,
                     const uint64_t* seed_dev /* nullable: *seed_dev is added to seed */,
                     int nrep /* 1: sum / sumsq are the batch sums; n > 1: n replicas [sum[C] | sumsq[C]] (stride 2C doubles from
                                 `sum` resp. `sumsq`) whose sum they are, as uaps_conv_fprop_bn leaves them */,
                     cudaStream_t stream);
int uaps_bn_act_bwd_nhwc(const void* g_out, const void* y, const float* gamma, const float* beta,
                         const float* save_mean, const float* save_rstd, float slope, double p_drop,
                         uint64_t seed, double* sum_g, double* sum_gx, void* dy,
                         float* dgamma_accum, float* dbeta_accum, /* nullable pair: fp32 [C], += d gamma / d beta */
                         int64_t npix, int C, const uint64_t* seed_dev, cudaStream_t stream);

/* ---------------------------------------------------------------------------------------------
 * Implicit-GEMM convolution on tcgen05 / TMEM / TMA (3x3 pad 1 or 1x1, stride 1), bf16 operands, fp32
 * accumulation.  Replaces the cuDNN calls behind nn.Conv2d in utilities/UAPS_unet.py:36,41 (ConvBlock),
 * :73 (UpBlock conv1x1), :138 (out_conv) and, with transpose = 1 packing, their data gradients.
 * Activations: NHWC bf16, channel pitch c*_stride (a multiple of 8 that covers the channel count
 * rounded up to 16; padding channels must be zero).  x2 (nullable, cin2 = 0) is a second K segment:
 * conv(cat([x1, x2], channel)) without materialising the concat (UAPS_unet.py:85).
 * Output: bf16 NHWC with channel pitch out_c_stride, or fp32 NCHW (out_nchw_f32 = 1, the layout the
 * fused loss kernel consumes).  bias: fp32 [cout] or NULL.
 * ------------------------------------------------------------------------------------------- */
/* fold = F in {1, 2, 4}: pixel folding.  F horizontally adjacent pixels of a small-channel tensor are viewed as
 * one pixel with F*C channels (the same memory); the kernel runs the equivalent convolution with F*Cin input and
 * F*Cout output channels and block-banded weights.  F times the MACs (these layers are bandwidth bound) for F
 * times wider TMA rows -- the 16/32-channel layers are otherwise limited by TMA's per-row rate.  Needs W % F == 0
 * and channel pitches equal to the channel counts rounded up to 16; all other arguments stay the REAL sizes. */
size_t uaps_conv_packed_bytes(int cout, int cin1, int cin2, int ks, int fold);
/* w: device fp32 in torch layout [cout][cin1+cin2][ks][ks]; transpose = 1 packs the data-gradient
 * kernel W'[ci][co][r][s] = W[co][ci][ks-1-r][ks-1-s] (then cout/cin name W's input/output channels
 * swapped: pass cout = W's Cin, cin1 = W's Cout). */
int uaps_conv_pack_weights(const float* w, void* w_packed, int cout, int cin1, int cin2, int ks,
                           int transpose, int fold, cudaStream_t stream);
/* All layers in one launch: a training iteration re-packs ~124 (layer, layout) pairs after every optimizer step; one launch
 * each costs 4-5 us.  uaps_conv_pack_plan turns a host job list into a HOST table of n_jobs records of
 * uaps_conv_pack_job_bytes() bytes; the caller copies the table to device memory once (the addresses in it -- parameters and
 * packed buffers -- must stay fixed); uaps_conv_pack_run re-packs every layer from the current weights with ONE launch. */
typedef struct UapsPackJob {
    const float* w;      /* device, torch layout [cout][cin1+cin2][ks][ks] (as uaps_conv_pack_weights) */
    void* w_packed;      /* device, uaps_conv_packed_bytes(...) bytes, 16-byte aligned                   */
    int cout, cin1, cin2, ks, transpose, fold;
} UapsPackJob;
size_t uaps_conv_pack_job_bytes(void);
int uaps_conv_pack_plan(const UapsPackJob* jobs, int n_jobs, void* table_host, int* total_blocks);
int uaps_conv_pack_run(const void* table_dev, int n_jobs, int total_blocks, cudaStream_t stream);
/* out2 (nullable): second bf16 NHWC output; output channels >= split (a multiple of 16) are written there
 * at channel (c - split) -- the data gradient of a concat convolution lands in its two consumers' tensors. */
int uaps_conv_fprop(const void* x1, int c1_stride, const void* x2, int c2_stride, const void* w_packed,
                    const float* bias, void* out, int out_c_stride, int out_nchw_f32,
                    int B, int H, int W, int cin1, int cin2, int cout, int ks,
                    void* out2, int out2_c_stride, int split, int fold, cudaStream_t stream);
/* conv + bias -> bf16 NHWC (as uaps_conv_fprop without out2 / fold / NCHW) AND the BatchNorm batch statistics of that
 * output from the accumulators, in the same kernel (utilities/UAPS_unet.py:36-38, 41-42: nn.Conv2d -> nn.BatchNorm2d):
 * saves the separate pass over the output that uaps_bn_stats_nhwc makes.  bn_sums: bn_nrep replicas of
 * [sum[out_c_stride] | sumsq[out_c_stride]] doubles, zeroed by the caller (replicas spread the per-CTA atomics);
 * hand them to uaps_bn_act_nhwc(sum = bn_sums, sumsq = bn_sums + out_c_stride, ..., nrep = bn_nrep). */
int uaps_conv_fprop_bn(const void* x1, int c1_stride, const void* x2, int c2_stride, const void* w_packed,
                       const float* bias, void* out, int out_c_stride, int B, int H, int W,
                       int cin1, int cin2, int cout, int ks, double* bn_sums, int bn_nrep, cudaStream_t stream);
/* The same with y = leaky_relu(conv(x) + bias, leaky_slope) in the epilogue (leaky_slope = 1: identity).  With the
 * running statistics of the following BatchNorm2d folded into weights and bias, one call is a whole eval-mode
 * conv -> BN -> LeakyReLU layer of ConvBlock (utilities/UAPS_unet.py:36-43): the validation / inference forward
 * of UAPS_train.py:367-393. */
int uaps_conv_fprop_act(const void* x1, int c1_stride, const void* x2, int c2_stride, const void* w_packed,
                        const float* bias, void* out, int out_c_stride, int out_nchw_f32, int B, int H, int W,
                        int cin1, int cin2, int cout, int ks, void* out2, int out2_c_stride, int split,
                        int fold, float leaky_slope, cudaStream_t stream);

/* Weight gradient on tcgen05 (MN-major operands straight from the channels-last tensors):
 * dw[co][ci_offset + ci][r][s] += sum_pixels dy[p][co] * x[p + (r-1, s-1)][ci].  dw is fp32 in torch layout
 * [cout][cin_total][ks][ks] and is ACCUMULATED into (zero it first); a concatenated input is two calls
 * with different ci_offset.  cin must be a multiple of 16 (pad the 3-channel network input).
 * workspace (nullable): deterministic split-K.  The pixel dimension is split over CTAs; without a workspace their partial
 * sums meet in dw through fp32 atomics (cout*cin*ks*ks of them per split: half the kernel's time on the 64..256-channel
 * layers, and a run-to-run rounding order).  With >= uaps_conv_wgrad_workspace_bytes of 16-byte-aligned scratch whose first
 * 256 bytes are zero before the first use (every launch leaves them zero), the CTAs store their partials, meet at a grid
 * barrier (the launch is one co-resident wave) and fold them in split order: no atomics, bit-reproducible.  The same
 * scratch can serve every call of a stream (the fold ends inside the launch). */
size_t uaps_conv_wgrad_workspace_bytes(int B, int H, int W, int cout, int cin, int ks);
int uaps_conv_wgrad(const void* dy, int dy_c_stride, const void* x, int x_c_stride, float* dw,
                    int B, int H, int W, int cout, int cin, int cin_total, int ci_offset, int ks,
                    void* workspace, size_t workspace_bytes, cudaStream_t stream);

/* ---- optimizer (UAPS_train.py:112, 292: torch.optim.Adam(model.parameters(), lr) and its step()) -----------------
 * One Adam step over flat fp32 buffers of n elements (parameters, gradients, first and second moments; 16-byte
 * aligned): torch's update rule with its defaults' structure (no weight decay, no amsgrad):
 *   m = b1 m + (1-b1) g;  v = b2 v + (1-b2) g^2;  p -= lr/(1-b1^step) * m / (sqrt(v)/sqrt(1-b2^step) + eps).
 * step = 1, 2, 3, ...; grad_scale multiplies g first (1 when the gradient is already that of the global loss). */
int uaps_adam_step(float* p, const float* g, float* m, float* v, int64_t n, int64_t step, float lr, float beta1,
                   float beta2, float eps, float grad_scale,
                   UapsStepState* state,   /* nullable: step size / bias correction come from the device state (step, lr ignored) */
                   const float* guard,     /* nullable device float (the iteration's loss): if it is not finite the update is
                                              skipped and state->skipped / n_skipped record it (needs state) */
                   cudaStream_t stream);

/* ---- gradient all-reduce fused with the Adam step, over NVLink peer memory ------------------------------------------
 * (replaces the gradient sum of nn.DataParallel, UAPS_model.py:13, plus optimizer_1.step(), UAPS_train.py:292, at N > 1.)
 * Every rank's flat gradient buffer lives in a peer-mappable allocation (uaps_peer_alloc; exported / mapped / unmapped
 * with uaps_xchg_export / _import / _close).  ONE kernel per rank: wait until every rank's gradients are complete, read
 * all ranks' gradients (peers' over NVLink) and add them in rank order -- bit-identical sums on every rank --, apply the
 * Adam update to the local replica, wait until every rank has finished reading.  No NCCL call, so the iteration stays a
 * capturable kernel sequence.  grads / flagboxes: host arrays of `world` device pointers as mapped in THIS process (own at
 * [rank]); a flag box is a zero-initialised uaps_xchg_alloc mailbox used only for this purpose.  The other arguments are
 * those of uaps_adam_step.  n must be a multiple of 4.  Waits are bounded by UAPS_XCHG_TIMEOUT_MS (default 30000): on a
 * time-out the update is skipped and word 81 of the own flag box latches the epoch. */
int uaps_peer_alloc(void** ptr, size_t bytes);
int uaps_peer_free(void* ptr);
int uaps_grad_reduce_adam(float* p, const float* const* grads, float* m, float* v, int64_t n,
                          void* const* flagboxes, int rank, int world, int64_t step, float lr, float beta1,
                          float beta2, float eps, float grad_scale, UapsStepState* state, const float* guard,
                          cudaStream_t stream);

/* On-device confusion matrix behind utilities/metrics.py (pixel_accuracy :8, mIoU :16, mDice :40):
 * conf[label * C + argmax(softmax(logits))] += 1 per pixel (labels outside [0,C) ignored).  logits [B,C,HW] fp32,
 * labels [B,HW] int64, conf C*C uint64 ACCUMULATED into. */
int uaps_confusion(const float* logits, const int64_t* labels, int B, int C, int64_t HW, uint64_t* conf,
                   cudaStream_t stream);

/* ---------------------------------------------------------------------------------------------
 * Validation head: one validation batch of UAPS_train.py:377-385 (main decoder's logits -> CrossEntropyLoss() with
 * torch's default ignore_index -100, and the confusion matrix behind utilities/metrics.py), appended as one row of an
 * epoch table that stays on the device until the epoch ends.
 *   uaps_val_counts: reads logits [B,C,HW] fp32 and labels [B,HW] int64 once; per pixel pred = argmax(softmax(z))
 *     (bit-exact with torch, as uaps_confusion) and the fp32 term -log_softmax(z)[y].  A label of -100 is left out of the
 *     CE and the counts (it still counts as a pixel); any other label outside [0, C) is counted as BAD.  Per-block partial
 *     sums go to `workspace` (>= uaps_val_workspace_bytes(C, B, HW) bytes, 8-byte aligned, no initialisation needed).
 *   uaps_val_fold: one block adds those partials in a fixed order (bitwise reproducible) and writes row r = state[0] of
 *     table[max_batches][C*C + 3] (fp64): C*C counts (row = label, column = prediction) | CE sum over the non-ignored
 *     pixels | non-ignored pixels | pixels (B*HW); then state[0] = r + 1.  If r >= max_batches nothing is written and
 *     state[1] = 1 (overflow).  state[2] += the batch's bad labels.  state: 3 uint32, zeroed by the caller per table.
 * Same (B, C, HW) and workspace in both calls.  Both only read and write device memory at addresses fixed by their
 * arguments, so the pair can be captured into a CUDA graph: every replay appends the next row.
 * Algorithmic HBM bytes per pixel: 4C (logits) + 8 (label) read.
 * ------------------------------------------------------------------------------------------- */
size_t uaps_val_workspace_bytes(int C, int B, int64_t HW);
int uaps_val_counts(const float* logits, const int64_t* labels, int B, int C, int64_t HW, void* workspace,
                    size_t workspace_bytes, cudaStream_t stream);
int uaps_val_fold(const void* workspace, size_t workspace_bytes, int B, int C, int64_t HW, double* table,
                  int max_batches, uint32_t* state, cudaStream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* UAPS_B200_H */
