"""Host-side contract of the ensemble inference path (no GPU needed): argument checks, the seed-derived draws, the
C ABI's workspace query and its validation of arguments before any launch."""
import ctypes

import numpy as np
import pytest
import torch


def test_ensemble_uncertainty_refuses_cpu_tensors():
    from uaps_b200.ensemble import ensemble_uncertainty
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        ensemble_uncertainty([torch.randn(1, 4, 8, 8) for _ in range(3)])


def test_predict_uncertainty_argument_checks():
    from uaps_b200.unet import UNet_UAPS
    with pytest.raises(ValueError, match="auxiliary decoder"):
        UNet_UAPS(3, 4, n_aux=0).eval().predict_uncertainty(torch.randn(1, 3, 32, 32))
    m = UNet_UAPS(3, 4, n_aux=3).eval()
    for shape in ((1, 3, 40, 32), (1, 3, 32, 24)):
        with pytest.raises(RuntimeError, match="multiples of 16"):
            m.predict_uncertainty(torch.randn(*shape))
        with pytest.raises(RuntimeError, match="multiples of 16"):
            m.predict_uncertainty_graphed(torch.randn(*shape))


@pytest.mark.parametrize("n_aux", [1, 3, 4, 5])
def test_seed_derived_draws_follow_the_documented_order(n_aux):
    from uaps_b200.unet import UNet_UAPS
    m = UNet_UAPS(3, 2, n_aux=n_aux)
    n = 5 * (1 + max(0, n_aux - 3))
    got = m._ensemble_draws(1234)
    assert got.shape == (2, n) and got.dtype == np.int64
    rng = np.random.default_rng(1234)                      # predict_uncertainty's docstring: key_i, then u_i, per launch
    for i in range(n):
        key, u = rng.integers(0, 2 ** 63 - 1), rng.uniform(0.7, 0.9)
        assert got[0, i] == key
        assert got[1, i:i + 1].view(np.float32)[0] == np.float32(u)
    assert np.array_equal(m._ensemble_draws(1234), got)
    assert not np.array_equal(m._ensemble_draws(1235), got)


def test_ensemble_abi_host_checks():
    from uaps_b200 import _lib as L
    lib = L.lib()
    assert lib.uaps_ensemble_workspace_bytes(4, 4, 64, 65536) == 64 * 512 * 8
    assert lib.uaps_ensemble_workspace_bytes(4, 4, 2, 63) == 2 * 1 * 8
    for bad in ((7, 4), (0, 4), (4, 9), (4, 1)):
        assert lib.uaps_ensemble_workspace_bytes(*bad, 1, 64) == 0
    fake = ctypes.c_void_p(4096)                            # never dereferenced: every call below fails its checks first
    z = L.ptr_array([None] * 4)
    z_ok = (ctypes.c_void_p * 7)(*([4096] * 7))
    assert lib.uaps_ensemble_head(None, 4, 1, 4, 64, fake, None, None, None, None, 0, None) == -1
    assert lib.uaps_ensemble_head(z, 4, 1, 4, 64, fake, None, None, None, None, 0, None) == -1
    assert lib.uaps_ensemble_head(z_ok, 7, 1, 4, 64, fake, None, None, None, None, 0, None) == -2
    assert lib.uaps_ensemble_head(z_ok, 4, 1, 9, 64, fake, None, None, None, None, 0, None) == -2
    assert lib.uaps_ensemble_head(z_ok, 4, 1, 4, 64, None, None, None, None, None, 0, None) == -1
    assert lib.uaps_ensemble_head(z_ok, 4, 1, 4, 64, fake, ctypes.c_void_p(4098), None, None, None, 0, None) == -3
    # the per-image mean needs a workspace large enough for the launch's chunks
    assert lib.uaps_ensemble_head(z_ok, 4, 1, 4, 64, fake, None, fake, None, None, 0, None) == -1
    assert lib.uaps_ensemble_head(z_ok, 4, 1, 4, 64, fake, None, fake, None, fake, 0, None) == -1
