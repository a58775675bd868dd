"""Host side of ensemble uncertainty inference through the C ABI (no GPU needed): exports, the parameter blob that
``uaps_b200.unet.inference_params(..., ensemble=True)`` builds against ``uaps_unet_ensemble_params_count``, the draws
count, the size queries, the layer offsets, and every argument check of prepare / run, which all come before any
launch."""
import ctypes

import pytest
import torch

NEW = ("uaps_unet_ensemble_params_count", "uaps_unet_ensemble_state_bytes", "uaps_unet_ensemble_draws_count",
       "uaps_unet_ensemble_workspace_bytes", "uaps_unet_ensemble_prepare", "uaps_unet_ensemble_run",
       "uaps_unet_ensemble_layer")


def test_exports():
    from uaps_b200 import _lib as L
    handle = ctypes.CDLL(L.LIB_PATH)
    for name in NEW:
        assert hasattr(handle, name) and name in L.exported_symbols()


def _decoder_floats(sd, prefix):
    return sum(v.numel() for k, v in sd.items() if k.startswith(prefix) and not k.endswith("num_batches_tracked"))


@pytest.mark.parametrize("n_aux", [1, 2, 3, 4, 5])
@pytest.mark.parametrize("C", [2, 4, 7])
@pytest.mark.parametrize("cin", [1, 3])
def test_params_count_is_the_blob_length(cin, C, n_aux):
    from uaps_b200 import _lib as L
    from uaps_b200.unet import UNet_UAPS, inference_params
    model = UNet_UAPS(cin, C, n_aux=n_aux)
    blob = inference_params(model, ensemble=True)
    assert blob.dtype == torch.float32 and blob.is_contiguous() and blob.dim() == 1
    lib = L.lib()
    assert lib.uaps_unet_ensemble_params_count(cin, C, n_aux) == blob.numel()
    one_decoder = _decoder_floats(model.state_dict(), "main_decoder.")
    assert blob.numel() == lib.uaps_unet_params_count(cin, C) + n_aux * one_decoder
    # the default blob is the f7 one, and the ensemble blob starts with it
    default = inference_params(model)
    assert default.numel() == lib.uaps_unet_params_count(cin, C)
    assert torch.equal(blob[:default.numel()], default)


def test_blob_follows_state_dict_order_and_accepts_the_module_prefix():
    from uaps_b200.unet import UNet_UAPS, inference_params
    model = UNet_UAPS(3, 4, n_aux=4)
    with torch.no_grad():
        for i, t in enumerate(model.state_dict().values()):     # every tensor gets values that name it
            if t.is_floating_point():
                t.copy_(torch.arange(t.numel(), dtype=t.dtype).view_as(t) * 1e-3 + i)
    sd = model.state_dict()
    blob = inference_params(model, ensemble=True)
    off = 0
    for k, v in sd.items():
        if k.endswith("num_batches_tracked"):
            continue
        assert torch.equal(blob[off:off + v.numel()], v.reshape(-1)), k
        off += v.numel()
    assert off == blob.numel()
    ref_ck = {"module." + k: v for k, v in sd.items()}               # a reference (DataParallel) checkpoint
    assert torch.equal(inference_params(ref_ck, ensemble=True), blob)
    # the default blob still leaves the auxiliary decoders out
    want = torch.cat([v.reshape(-1) for k, v in sd.items()
                      if k.startswith(("encoder.", "main_decoder.")) and not k.endswith("num_batches_tracked")])
    assert torch.equal(inference_params(ref_ck), want)


def test_blob_rejects_missing_or_gapped_auxiliary_decoders():
    from uaps_b200.unet import UNet_UAPS, inference_params
    with pytest.raises(ValueError, match="auxiliary decoders"):
        inference_params(UNet_UAPS(3, 4, n_aux=0), ensemble=True)
    sd = UNet_UAPS(3, 4, n_aux=3).state_dict()
    gap = {k: v for k, v in sd.items() if not k.startswith("aux_decoder2.")}
    with pytest.raises(ValueError, match="auxiliary decoders"):
        inference_params(gap, ensemble=True)
    six = dict(UNet_UAPS(3, 4, n_aux=5).state_dict())
    six.update({k.replace("aux_decoder5.", "aux_decoder6."): v for k, v in six.items() if k.startswith("aux_decoder5.")})
    with pytest.raises(ValueError, match="auxiliary decoders"):
        inference_params(six, ensemble=True)
    short = dict(sd)
    del short["aux_decoder3.out_conv.bias"]
    with pytest.raises(ValueError, match="needs"):
        inference_params(short, ensemble=True)


@pytest.mark.parametrize("n_aux", [1, 2, 3, 4, 5])
def test_draws_count(n_aux):
    from uaps_b200 import _lib as L
    from uaps_b200.unet import UNet_UAPS
    assert L.lib().uaps_unet_ensemble_draws_count(n_aux) == UNet_UAPS(3, 4, n_aux=n_aux)._ensemble_calls()


def test_size_queries():
    from uaps_b200 import _lib as L
    lib = L.lib()
    for cin, C, n_aux in ((1, 2, 1), (3, 4, 3), (3, 2, 4), (16, 8, 5)):
        assert lib.uaps_unet_ensemble_state_bytes(cin, C, n_aux) > 4 * lib.uaps_unet_ensemble_params_count(cin, C, n_aux) > 0
        assert lib.uaps_unet_ensemble_state_bytes(cin, C, n_aux) > lib.uaps_unet_infer_state_bytes(cin, C)
        sizes = [lib.uaps_unet_ensemble_workspace_bytes(cin, C, n_aux, B, H, W)
                 for B, H, W in ((1, 16, 16), (1, 64, 64), (2, 64, 64), (2, 64, 128), (64, 256, 256))]
        assert all(s > 0 for s in sizes) and sizes == sorted(sizes) and len(set(sizes)) == len(sizes)
        # per pixel: 126 (encoder maps + scratch) + 62 per perturbed copy + 4 C per decoder's logits (+ 4, attention)
        per_px = 126 + 62 * min(n_aux, 3) + 4 * C * (1 + n_aux) + (4 if n_aux >= 3 else 0)
        assert per_px * 64 * 256 * 256 < sizes[-1] < (per_px + 1) * 64 * 256 * 256
    for cin, C, n_aux in ((0, 4, 3), (17, 4, 3), (3, 1, 3), (3, 9, 3), (3, 4, 0), (3, 4, 6)):
        assert lib.uaps_unet_ensemble_params_count(cin, C, n_aux) == 0
        assert lib.uaps_unet_ensemble_state_bytes(cin, C, n_aux) == 0
        assert lib.uaps_unet_ensemble_workspace_bytes(cin, C, n_aux, 1, 64, 64) == 0
    for n_aux in (0, 6, -1):
        assert lib.uaps_unet_ensemble_draws_count(n_aux) == 0
    for B, H, W in ((0, 64, 64), (1, 0, 64), (1, 56, 64), (1, 64, 40), (65536, 16, 16)):
        assert lib.uaps_unet_ensemble_workspace_bytes(3, 4, 3, B, H, W) == 0


@pytest.mark.parametrize("n_aux", [1, 3, 5])
def test_layer_offsets(n_aux):
    from uaps_b200 import _lib as L
    lib = L.lib()
    o = [ctypes.c_size_t() for _ in range(4)]
    refs = [ctypes.byref(v) for v in o]
    n_layers = 23 + 13 * n_aux
    end = 0
    for layer in range(n_layers):
        assert lib.uaps_unet_ensemble_layer(3, 4, n_aux, layer, *refs) == 0
        w, b, p, n = (v.value for v in o)
        assert w % 256 == 0 and b % 256 == 0 and p % 256 == 0 and n > 0 and end <= w < b < p
        end = p + n
    assert end <= lib.uaps_unet_ensemble_state_bytes(3, 4, n_aux)
    # an auxiliary decoder's layer has the shape of the main decoder's layer at the same position
    for layer in range(23, n_layers):
        main = (layer - 23) % 13 + 10
        assert lib.uaps_unet_ensemble_layer(3, 4, n_aux, layer, *refs) == 0
        aux_n = o[3].value
        assert lib.uaps_unet_ensemble_layer(3, 4, n_aux, main, *refs) == 0
        assert o[3].value == aux_n
    assert lib.uaps_unet_ensemble_layer(3, 4, n_aux, n_layers, *refs) == -2
    assert lib.uaps_unet_ensemble_layer(3, 4, n_aux, -1, *refs) == -2
    assert lib.uaps_unet_ensemble_layer(3, 9, n_aux, 0, *refs) == -2
    assert lib.uaps_unet_ensemble_layer(3, 4, 0, 0, *refs) == -2
    assert lib.uaps_unet_ensemble_layer(3, 4, 6, 0, *refs) == -2
    assert lib.uaps_unet_ensemble_layer(3, 4, n_aux, 0, None, *refs[1:]) == -1


def test_argument_checks():
    from uaps_b200 import _lib as L
    lib = L.lib()
    fake, odd, odd4, odd8 = (ctypes.c_void_p(a) for a in (4096, 4098, 4100, 4104))   # never dereferenced
    sb = lib.uaps_unet_ensemble_state_bytes(3, 4, 3)
    wb = lib.uaps_unet_ensemble_workspace_bytes(3, 4, 3, 2, 64, 64)

    def prep(params=fake, cin=3, C=4, n_aux=3, state=fake, nbytes=sb):
        return lib.uaps_unet_ensemble_prepare(params, cin, C, n_aux, state, nbytes, None)

    assert prep(params=None) == -1 and prep(state=None) == -1
    assert prep(cin=0) == -2 and prep(cin=17) == -2 and prep(C=1) == -2 and prep(C=9) == -2
    assert prep(n_aux=0) == -2 and prep(n_aux=6) == -2
    assert prep(params=odd) == -3 and prep(state=odd4) == -3
    assert prep(nbytes=sb - 1) == -1

    def run(state=fake, sbytes=sb, cin=3, C=4, n_aux=3, x=fake, B=2, H=64, W=64, draws=fake, ws=fake, wbytes=wb,
            labels=fake, unc=fake, img=fake, prob=fake):
        return lib.uaps_unet_ensemble_run(state, sbytes, cin, C, n_aux, x, B, H, W, draws, ws, wbytes, labels, unc, img,
                                          prob, None)

    for kw in ({"state": None}, {"x": None}, {"draws": None}, {"ws": None}, {"labels": None}):
        assert run(**kw) == -1, kw
    assert run(B=0) == -1 and run(H=0) == -1 and run(W=-16) == -1
    assert run(H=56) == -2 and run(W=72) == -2 and run(B=65536) == -2
    assert run(cin=0) == -2 and run(cin=17) == -2 and run(C=1) == -2 and run(C=9) == -2
    assert run(n_aux=0) == -2 and run(n_aux=6) == -2
    for kw in ({"state": odd4}, {"x": odd4}, {"draws": odd4}, {"ws": odd8}, {"labels": odd}, {"unc": odd4},
               {"img": odd4}, {"prob": odd8}):
        assert run(**kw) == -3, kw
    assert run(sbytes=sb - 1) == -1 and run(wbytes=wb - 1) == -1
    assert run(wbytes=lib.uaps_unet_ensemble_workspace_bytes(3, 4, 3, 1, 64, 64), B=2) == -1
    assert run(sbytes=lib.uaps_unet_infer_state_bytes(3, 4)) == -1                 # an f7 state is too small
    assert run(n_aux=4, wbytes=lib.uaps_unet_ensemble_workspace_bytes(3, 4, 3, 2, 64, 64),
               sbytes=lib.uaps_unet_ensemble_state_bytes(3, 4, 4)) == -1           # workspace sized for fewer decoders
