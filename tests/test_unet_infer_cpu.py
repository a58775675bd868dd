"""Host side of whole-network inference through the C ABI (no GPU needed): exports, the parameter blob that
``uaps_b200.unet.inference_params`` builds against ``uaps_unet_params_count``, the size queries, and every argument
check of prepare / run, which all come before any launch."""
import ctypes

import pytest
import torch

NEW = ("uaps_unet_params_count", "uaps_unet_infer_state_bytes", "uaps_unet_infer_workspace_bytes",
       "uaps_unet_infer_prepare", "uaps_unet_infer_run", "uaps_unet_infer_layer")


def test_exports():
    from uaps_b200 import _lib as L
    handle = ctypes.CDLL(L.LIB_PATH)
    for name in NEW:
        assert hasattr(handle, name) and name in L.exported_symbols()


@pytest.mark.parametrize("cin", [1, 3])
@pytest.mark.parametrize("C", [2, 4, 7])
def test_params_count_is_the_blob_length(cin, C):
    from uaps_b200 import _lib as L
    from uaps_b200.unet import UNet_UAPS, inference_params
    model = UNet_UAPS(cin, C)
    blob = inference_params(model)
    assert blob.dtype == torch.float32 and blob.is_contiguous() and blob.dim() == 1
    assert L.lib().uaps_unet_params_count(cin, C) == blob.numel()
    # the auxiliary decoders are left out: the count does not depend on them
    assert inference_params(UNet_UAPS(cin, C, n_aux=0)).numel() == blob.numel()


def test_blob_follows_state_dict_order_and_accepts_the_module_prefix():
    from uaps_b200.unet import UNet_UAPS, inference_params
    model = UNet_UAPS(3, 4)
    with torch.no_grad():
        for i, t in enumerate(model.state_dict().values()):     # every tensor gets values that name it
            if t.is_floating_point():
                t.copy_(torch.arange(t.numel(), dtype=t.dtype).view_as(t) * 1e-3 + i)
    sd = model.state_dict()
    blob = inference_params(model)
    off = 0
    for k, v in sd.items():
        if not k.startswith(("encoder.", "main_decoder.")) or k.endswith("num_batches_tracked"):
            continue
        assert torch.equal(blob[off:off + v.numel()], v.reshape(-1)), k
        off += v.numel()
    assert off == blob.numel()
    ref_ck = {"module." + k: v for k, v in sd.items()}               # a reference (DataParallel) checkpoint
    assert torch.equal(inference_params(ref_ck), blob)


def test_blob_rejects_a_foreign_state_dict():
    from uaps_b200.unet import UNet_UAPS, inference_params
    sd = UNet_UAPS(3, 4).state_dict()
    del sd["encoder.in_conv.conv_conv.1.running_var"]
    with pytest.raises(ValueError, match="needs"):
        inference_params(sd)
    with pytest.raises(ValueError, match="missing"):
        inference_params({"encoder.x": torch.zeros(1)})


def test_size_queries():
    from uaps_b200 import _lib as L
    lib = L.lib()
    for cin, C in ((1, 2), (3, 4), (16, 8)):
        assert lib.uaps_unet_infer_state_bytes(cin, C) > 4 * lib.uaps_unet_params_count(cin, C) > 0
        sizes = [lib.uaps_unet_infer_workspace_bytes(cin, C, B, H, W)
                 for B, H, W in ((1, 16, 16), (1, 64, 64), (2, 64, 64), (2, 64, 128), (64, 256, 256))]
        assert all(s > 0 for s in sizes) and sizes == sorted(sizes) and len(set(sizes)) == len(sizes)
        # about 126 bytes per pixel: five encoder maps + two scratch buffers
        assert 120 * 64 * 256 * 256 < sizes[-1] < 130 * 64 * 256 * 256
    for cin, C in ((0, 4), (17, 4), (3, 1), (3, 9)):
        assert lib.uaps_unet_params_count(cin, C) == 0 and lib.uaps_unet_infer_state_bytes(cin, C) == 0
        assert lib.uaps_unet_infer_workspace_bytes(cin, C, 1, 64, 64) == 0
    for B, H, W in ((0, 64, 64), (1, 0, 64), (1, 56, 64), (1, 64, 40), (65536, 16, 16)):
        assert lib.uaps_unet_infer_workspace_bytes(3, 4, B, H, W) == 0


def test_layer_offsets():
    from uaps_b200 import _lib as L
    lib = L.lib()
    o = [ctypes.c_size_t() for _ in range(4)]
    refs = [ctypes.byref(v) for v in o]
    end = 0
    for layer in range(23):
        assert lib.uaps_unet_infer_layer(3, 4, layer, *refs) == 0
        w, b, p, n = (v.value for v in o)
        assert w % 256 == 0 and b % 256 == 0 and p % 256 == 0 and n > 0 and end <= w < b < p
        end = p + n
    assert end <= lib.uaps_unet_infer_state_bytes(3, 4)
    assert lib.uaps_unet_infer_layer(3, 4, 23, *refs) == -2
    assert lib.uaps_unet_infer_layer(3, 4, -1, *refs) == -2
    assert lib.uaps_unet_infer_layer(3, 9, 0, *refs) == -2
    assert lib.uaps_unet_infer_layer(3, 4, 0, None, *refs[1:]) == -1


def test_argument_checks():
    from uaps_b200 import _lib as L
    lib = L.lib()
    fake, odd, odd4 = ctypes.c_void_p(4096), ctypes.c_void_p(4098), ctypes.c_void_p(4100)   # never dereferenced
    sb = lib.uaps_unet_infer_state_bytes(3, 4)
    wb = lib.uaps_unet_infer_workspace_bytes(3, 4, 2, 64, 64)

    def prep(params=fake, cin=3, C=4, state=fake, nbytes=sb):
        return lib.uaps_unet_infer_prepare(params, cin, C, state, nbytes, None)

    assert prep(params=None) == -1 and prep(state=None) == -1
    assert prep(cin=0) == -2 and prep(cin=17) == -2 and prep(C=1) == -2 and prep(C=9) == -2
    assert prep(params=odd) == -3 and prep(state=odd4) == -3
    assert prep(nbytes=sb - 1) == -1

    def run(state=fake, sbytes=sb, cin=3, C=4, x=fake, B=2, H=64, W=64, ws=fake, wbytes=wb, logits=fake, labels=fake):
        return lib.uaps_unet_infer_run(state, sbytes, cin, C, x, B, H, W, ws, wbytes, logits, labels, None)

    assert run(state=None) == -1 and run(x=None) == -1 and run(ws=None) == -1
    assert run(logits=None, labels=None) == -1
    assert run(B=0) == -1 and run(H=0) == -1 and run(W=-16) == -1
    assert run(H=56) == -2 and run(W=72) == -2 and run(B=65536) == -2
    assert run(cin=0) == -2 and run(cin=17) == -2 and run(C=1) == -2 and run(C=9) == -2
    for kw in ({"state": odd4}, {"x": odd4}, {"ws": odd4}, {"logits": odd4}, {"labels": odd}):
        assert run(**kw) == -3, kw
    assert run(sbytes=sb - 1) == -1 and run(wbytes=wb - 1) == -1
    assert run(wbytes=lib.uaps_unet_infer_workspace_bytes(3, 4, 1, 64, 64), B=2) == -1
