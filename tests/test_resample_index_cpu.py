"""The two index invariants the bilinear x2 upsampling kernels of resample_nhwc.cu rely on, checked for every input size up
to 8192 with the kernels' own fp32 arithmetic (src_coord: s = r * o with r = (n - 1) / (2n - 1) rounded to fp32,
i0 = min((int)s, n - 1), i1 = i0 + (i0 < n - 1), weight of i1 = s - i0):

* forward: the upper tap of output row 2k + 1 is one of the two taps of row 2k, so three horizontally interpolated input
  rows serve both output rows of a thread;
* backward: every output o that reaches input i with a nonzero weight lies in [2i - 1, 2i + 2], the four candidates the
  gather kernel visits per axis.
"""
import numpy as np

NMAX = 8192


def _taps(n):
    r = np.float32(n - 1) / np.float32(2 * n - 1) if n > 1 else np.float32(0)
    o = np.arange(2 * n)
    s = r * o.astype(np.float32)
    assert s.dtype == np.float32
    i0 = np.minimum(s.astype(np.int64), n - 1)
    i1 = i0 + (i0 < n - 1)
    l1 = s - i0.astype(np.float32)
    return o, i0, i1, l1


def test_second_row_upper_tap_is_a_first_row_tap():
    for n in range(1, NMAX + 1):
        _, i0, i1, _ = _taps(n)
        up_b = i0[1::2]
        bad = np.nonzero((up_b != i0[0::2]) & (up_b != i1[0::2]))[0]
        assert bad.size == 0, (n, bad[:8].tolist())


def test_backward_candidates_cover_every_weighted_tap():
    for n in range(1, NMAX + 1):
        o, i0, i1, l1 = _taps(n)
        w0 = np.float32(1) - l1
        out0 = ((o < 2 * i0 - 1) | (o > 2 * i0 + 2)) & (w0 != 0)
        out1 = ((o < 2 * i1 - 1) | (o > 2 * i1 + 2)) & (l1 != 0)
        assert not out0.any() and not out1.any(), (n, np.nonzero(out0 | out1)[0][:8].tolist())
        assert np.all((i0 >= 0) & (i1 <= n - 1))
