"""The host Philox oracle (oracle/philox_ref.py) against output words of the project's own Philox::draw4
(uaps_b200/csrc/common.cuh) compiled for the host, and its mask / noise derivations against their definitions."""
import numpy as np
import pytest

from oracle import philox_ref as R


@pytest.mark.parametrize("seed,idx,stream,words", [
    (0, 0, 0, "6627e8d5 e169c58d bc57ac4c 9b00dbd8"),             # also the published Random123 known-answer vector
    (0x0123456789ABCDEF, 0, 21, "086fe390 91d911c7 6d2095da 793484c5"),
    (0x9E3779B97F4A7C15, 123456789012, 11, "976ca40d d30a4e8a 2d1866d7 63e21237"),
    (2 ** 64 - 1, 2 ** 64 - 1, 12, "885511dd e940da8e 8d0409b6 18a29a97"),
])
def test_draw4_matches_device_words(seed, idx, stream, words):
    got = R.draw4(seed, [idx], stream)[0]
    assert " ".join(f"{int(v):08x}" for v in got) == words
    # vectorised draws equal one-at-a-time draws
    many = R.draw4(seed, [idx, 0, 7], stream)
    assert np.array_equal(many[0], got) and np.array_equal(many[2], R.draw4(seed, [7], stream)[0])


def test_seed_is_taken_mod_2_64():
    assert np.array_equal(R.draw4(2 ** 64 + 5, [3], 21), R.draw4(5, [3], 21))
    assert np.array_equal(R.draw4(-1, [3], 21), R.draw4(2 ** 64 - 1, [3], 21))


def test_sixteen_bit_uniforms_take_low_then_high_halves():
    seed, p = 99, 0.3
    w = R.draw4(seed, np.arange(4, dtype=np.uint64), R.STREAM_BN_DROP)         # npix = 1, C = 32: four chunks
    keep = R.bn_keep(seed, 1, 32, p)[0]
    for c in range(32):
        word = w[c // 8, (c % 8) // 2]
        u16 = (word & 0xFFFF) if c % 2 == 0 else (word >> 16)
        assert keep[c] == (u16 / 65536.0 >= float(np.float32(p)))


def test_nhwc_derivations():
    seed, B, hw, C, rng = 5, 3, 6, 16, 0.3
    n = R.nhwc_noise(seed, hw, C, rng)
    assert n.dtype == np.float32 and n.shape == (hw, C) and np.abs(n).max() <= np.float32(rng)
    w = R.draw4(seed, [1], R.STREAM_NHWC_NOISE)[0]                            # pixel 0, channels 8..15
    u = np.float32((w[1] >> 16) & 0xFFFF) / np.float32(65536.0)             # channel 8 + 3
    assert n[0, 11] == (u * np.float32(2) - np.float32(1)) * np.float32(rng)
    k = R.nhwc_keep(seed, B, hw, C, 0.5)
    assert k.shape == (B, hw, C) and not np.array_equal(k[0], k[1])
    w = R.draw4(seed, [(2 * hw + 4) * 2 + 1], R.STREAM_NHWC_DROP)[0]           # sample 2, pixel 4, channels 8..15
    assert k[2, 4, 8] == ((w[0] & 0xFFFF) / 65536.0 >= 0.5)


def test_nchw_derivations():
    seed = 17
    n = R.nchw_noise(seed, 10, 0.3)
    w = R.draw4(seed, [2], R.STREAM_NCHW_NOISE)[0]                            # element 9 = lane 1 of draw 2
    u = np.float32(w[1] >> 8) * np.float32(2.0 ** -24)
    assert n[9] == (u * np.float32(2) - np.float32(1)) * np.float32(0.3)
    k = R.nchw_keep(seed, 12, 0.25)
    w = R.draw4(seed, [2], R.STREAM_NCHW_DROP)[0]
    assert k[11] == (np.float32(w[3] >> 8) * np.float32(2.0 ** -24) >= np.float32(0.25))


@pytest.mark.parametrize("p", [0.05, 0.1, 0.2, 0.3, 0.5])
def test_keep_scale_rounds_like_the_kernels(p):
    assert R.keep_scale(p) == np.float32(1.0 / np.float64(np.float32(1.0 - p)))
    assert R.keep_scale(p).dtype == np.float32
