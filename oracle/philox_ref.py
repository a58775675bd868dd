"""Host restatement of the project's Philox4x32-10 and of every mask / noise derivation the kernels build on it.

``draw4`` is ``Philox::draw4`` (uaps_b200/csrc/common.cuh:150-156) in vectorised numpy: counter
``{idx_lo, idx_hi, stream, 0}``, key ``{seed_lo, seed_hi}``, ten rounds of ``Philox::round`` (:139-148).
The derivations below regenerate, bit for bit, what the CUDA kernels draw, so tests can compare dropout
masks and noise values exactly instead of statistically.  Layouts: channels-last tensors are indexed
``[pixel, C]`` (bf16 kernels), NCHW ones by the element index inside a sample (fp32 kernels).
"""
from __future__ import annotations

import numpy as np

M0, M1, W0, W1 = 0xD2511F53, 0xCD9E8D57, 0x9E3779B9, 0xBB67AE85
_M32 = np.uint64(0xFFFFFFFF)
MASK64 = (1 << 64) - 1

# stream ids (the third counter word) of each use
STREAM_NCHW_NOISE, STREAM_NCHW_DROP = 1, 2          # perturb.cu:21
STREAM_NHWC_NOISE, STREAM_NHWC_DROP = 11, 12        # perturb_nhwc.cu:15
STREAM_BN_DROP = 21                                 # bn_act_nhwc.cu:24


def draw4(seed: int, idx, stream: int) -> np.ndarray:
    """uint32 [..., 4]: the four output words of Philox4x32-10 for each counter index in ``idx``."""
    idx = np.asarray(idx, dtype=np.uint64)
    seed = int(seed) & MASK64
    c0, c1 = idx & _M32, idx >> np.uint64(32)
    c2 = np.full_like(idx, np.uint64(stream))
    c3 = np.zeros_like(idx)
    k0, k1 = np.uint64(seed & 0xFFFFFFFF), np.uint64(seed >> 32)
    m0, m1 = np.uint64(M0), np.uint64(M1)
    for _ in range(10):
        p0, p1 = m0 * c0, m1 * c2                   # exact: 32 x 32 -> 64 bits
        c0, c1, c2, c3 = (p1 >> np.uint64(32)) ^ c1 ^ k0, p1 & _M32, (p0 >> np.uint64(32)) ^ c3 ^ k1, p0 & _M32
        k0, k1 = (k0 + np.uint64(W0)) & _M32, (k1 + np.uint64(W1)) & _M32
    return np.stack([c0, c1, c2, c3], -1).astype(np.uint32)


def _u16x8(seed: int, chunk_idx, stream: int) -> np.ndarray:
    """float32 [..., 8]: the eight 16-bit uniforms of one draw, channel 2i from the low half of word i and channel 2i+1
    from the high half (perturb_nhwc.cu:31-39, bn_act_nhwc.cu:38-46); (u16) * 2^-16 is exact in fp32."""
    w = draw4(seed, chunk_idx, stream)
    u = np.empty(w.shape[:-1] + (8,), dtype=np.float32)
    u[..., 0::2] = (w & 0xFFFF).astype(np.float32)
    u[..., 1::2] = (w >> 16).astype(np.float32)
    return u * np.float32(1.0 / 65536.0)


def _chunks_nhwc(npix: int, C: int, base: int = 0) -> np.ndarray:
    """Counter index of each 16-byte chunk of a channels-last [npix, C] tensor: pixel * C/8 + c/8 (+ base)."""
    return np.arange(npix * (C // 8), dtype=np.uint64) + np.uint64(base)


def bn_keep(seed: int, npix: int, C: int, p: float) -> np.ndarray:
    """bool [npix, C]: the keep mask of the fused BatchNorm + LeakyReLU + Dropout kernels, stream 21, counter = the chunk
    index pixel * C/8 + c/8 (bn_act_nhwc.cu:183, :230, :287); kept iff u16 / 65536 >= float32(p) (:43-44)."""
    u = _u16x8(seed, _chunks_nhwc(npix, C), STREAM_BN_DROP)
    return (u >= np.float32(p)).reshape(npix, C)


def nhwc_noise(seed: int, hw: int, C: int, noise_range: float) -> np.ndarray:
    """float32 [hw, C]: the FeatureNoise draw of perturb3_nhwc, shared by every sample: stream 11, counter = the in-sample
    chunk index (perturb_nhwc.cu:112), value (u * 2 - 1) * float32(range) in fp32 (:114)."""
    u = _u16x8(seed, _chunks_nhwc(hw, C), STREAM_NHWC_NOISE)
    return ((u * np.float32(2.0) - np.float32(1.0)) * np.float32(noise_range)).reshape(hw, C)


def nhwc_keep(seed: int, B: int, hw: int, C: int, p: float) -> np.ndarray:
    """bool [B, hw, C]: the Dropout mask of perturb3_nhwc, stream 12, counter = the global chunk index
    b * hw * C/8 + pixel * C/8 + c/8 (perturb_nhwc.cu:118-120); kept iff u >= float32(p) (:137)."""
    u = _u16x8(seed, _chunks_nhwc(B * hw, C), STREAM_NHWC_DROP)
    return (u >= np.float32(p)).reshape(B, hw, C)


def _u01_nchw(seed: int, n: int, stream: int, base: int = 0) -> np.ndarray:
    """float32 [n]: element e (counted from ``base``) takes lane e % 4 of draw e / 4; u01 = (bits >> 8) * 2^-24
    (common.cuh:158)."""
    e = np.arange(n, dtype=np.uint64) + np.uint64(base)
    w = draw4(seed, e // np.uint64(4), stream)
    bits = np.take_along_axis(w, (e % np.uint64(4)).astype(np.int64)[:, None], axis=1)[:, 0]
    return (bits >> 8).astype(np.float32) * np.float32(1.0 / 16777216.0)


def nchw_noise(seed: int, chw: int, noise_range: float) -> np.ndarray:
    """float32 [chw]: the FeatureNoise draw of the fp32 kernels, stream 1, element e = c * HW + hw of a sample
    (perturb.cu:48-52, :180-182), value (u01 * 2 - 1) * float32(range) in fp32 (:27)."""
    u = _u01_nchw(seed, chw, STREAM_NCHW_NOISE)
    return (u * np.float32(2.0) - np.float32(1.0)) * np.float32(noise_range)


def nchw_keep(seed: int, n: int, p: float) -> np.ndarray:
    """bool [n]: the Dropout mask of the fp32 kernels, stream 2, element e = the global NCHW index (perturb.cu:78-80,
    :195-197); kept iff u01 >= float32(p) (:33)."""
    return _u01_nchw(seed, n, STREAM_NCHW_DROP) >= np.float32(p)


def keep_scale(p: float) -> np.float32:
    """1 / (1 - p) as every dropout kernel forms it: keep probability rounded to fp32, reciprocal in fp64, result to fp32
    (perturb.cu:213, bn_act_nhwc.cu:339, perturb_nhwc.cu:216)."""
    return np.float32(1.0 / float(np.float32(1.0 - p)))
