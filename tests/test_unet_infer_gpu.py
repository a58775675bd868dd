"""Whole-network inference through the C ABI on the B200: uaps_unet_infer_prepare folds and packs exactly what
UNet_UAPS._fold_bn / PackedConv produce, uaps_unet_infer_run returns UNet_UAPS.predict's logits bit for bit and torch's
argmax of the softmax as labels, inside a CUDA graph too, and examples/infer_c.c does the same with no Python."""
import ctypes
import os
import subprocess

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _model(cin, C, seed=0):
    """Eval-mode model whose BatchNorms carry non-trivial running statistics and affine parameters."""
    from uaps_b200.unet import UNet_UAPS
    torch.manual_seed(seed)
    model = UNet_UAPS(cin, C).cuda().eval()
    with torch.no_grad():
        for m in model.modules():
            if isinstance(m, torch.nn.BatchNorm2d):
                m.running_mean.normal_(0, 0.1)
                m.running_var.uniform_(0.5, 1.5)
                m.weight.normal_(1, 0.1)
                m.bias.normal_(0, 0.1)
    return model


class CInfer:
    """prepare + run over the raw entry points, on torch's current stream."""

    def __init__(self, model, cin, C):
        from uaps_b200 import _lib as L
        from uaps_b200.unet import inference_params
        self.L, self.lib, self.cin, self.C = L, L.lib(), cin, C
        self.state = torch.empty(self.lib.uaps_unet_infer_state_bytes(cin, C), dtype=torch.uint8, device="cuda")
        self.prepare(inference_params(model))

    def prepare(self, blob):
        self.L.check(self.lib.uaps_unet_infer_prepare(blob.data_ptr(), self.cin, self.C, self.state.data_ptr(),
                                                      self.state.numel(), self.L.stream_ptr()), "prepare")

    def run(self, x, logits=True, labels=True, out=None):
        B, _, H, W = x.shape
        ws = torch.empty(self.lib.uaps_unet_infer_workspace_bytes(self.cin, self.C, B, H, W), dtype=torch.uint8,
                         device="cuda")
        z, y = out if out is not None else (
            torch.empty(B, self.C, H, W, device="cuda") if logits else None,
            torch.empty(B, H, W, dtype=torch.uint8, device="cuda") if labels else None)
        self.L.check(self.lib.uaps_unet_infer_run(self.state.data_ptr(), self.state.numel(), self.cin, self.C, x.data_ptr(),
                                                  B, H, W, ws.data_ptr(), ws.numel(),
                                                  None if z is None else z.data_ptr(),
                                                  None if y is None else y.data_ptr(), self.L.stream_ptr()), "run")
        self.ws = ws
        return z, y


def _torch_labels(z):
    return torch.softmax(z, 1).argmax(1).to(torch.uint8)


def test_prepare_folds_and_packs_like_the_python_plan():
    from uaps_b200.conv import PackedConv
    from uaps_b200.unet import inference_params
    model = _model(3, 4)
    c = CInfer(model, 3, 4)
    # the packer writes only the bytes the selected kernel reads (the logits layer's conv_sn_small_kernel layout uses
    # 3 * C of its 16 rows per block and 3 of its 9 blocks): both packings go into zero-filled buffers
    c.state.zero_()
    c.prepare(inference_params(model))
    torch.cuda.synchronize()
    enc, dec, out = model._main_plan(make=lambda w, b, cin_split=None: (w, b, cin_split))
    layers = [l for blk in enc for l in blk] + [l for lvl in dec for l in lvl] + [out]
    assert len(layers) == 23
    state = c.state.cpu()
    o = [ctypes.c_size_t() for _ in range(4)]
    for i, (w, b, split) in enumerate(layers):
        assert c.lib.uaps_unet_infer_layer(3, 4, i, *[ctypes.byref(v) for v in o]) == 0
        w_off, b_off, p_off, p_n = (v.value for v in o)
        got_w = state[w_off:w_off + 4 * w.numel()].view(torch.float32).view_as(w)
        got_b = state[b_off:b_off + 4 * b.numel()].view(torch.float32)
        assert torch.equal(got_w, w.float().cpu()), f"layer {i} weight"
        assert torch.equal(got_b, b.float().cpu()), f"layer {i} bias"
        pc = PackedConv(w, b, cin_split=split)
        pc.packed.zero_()
        pc._pack(w.detach().float().contiguous())
        packed = pc.packed.cpu()
        assert p_n == packed.numel() and torch.equal(state[p_off:p_off + p_n], packed), f"layer {i} packed"


CASES = [(1, 3, 256, 256, 4), (4, 3, 64, 96, 4), (2, 1, 512, 512, 2), (2, 3, 240, 640, 2), (2, 3, 240, 640, 7)]


@pytest.mark.parametrize("B,cin,H,W,C", CASES)
def test_run_equals_predict(B, cin, H, W, C):
    model = _model(cin, C, seed=B + C)
    c = CInfer(model, cin, C)
    x = torch.randn(B, cin, H, W, device="cuda", generator=torch.Generator(device="cuda").manual_seed(7))
    z, y = c.run(x)
    want = model.predict(x)
    assert torch.equal(z, want)
    assert torch.equal(y, _torch_labels(want))


def test_labels_on_near_ties():
    """Classes 0 and 1 of out_conv differ by one ulp of the bias: their logits are (nearly) equal at every pixel, so
    softmax rounding decides, and torch then resolves equal probabilities to the lower index."""
    model = _model(3, 3, seed=5)
    with torch.no_grad():
        oc = model.main_decoder.out_conv
        oc.weight[1] = oc.weight[0]
        oc.bias[1] = torch.nextafter(oc.bias[0], torch.tensor(float("inf"), device="cuda"))
        oc.bias[2] = -10.0
    c = CInfer(model, 3, 3)
    x = torch.randn(2, 3, 64, 64, device="cuda")
    z, y = c.run(x)
    assert torch.equal(z, model.predict(x))
    assert ((z[:, 0] - z[:, 1]).abs() <= 1e-6).float().mean() > 0.9
    assert torch.equal(y, _torch_labels(z))


def test_labels_only_and_logits_only():
    """logits = NULL: the logits stay in the workspace and only the labels are written; labels = NULL: only logits."""
    model = _model(3, 4, seed=2)
    c = CInfer(model, 3, 4)
    x = torch.randn(2, 3, 64, 128, device="cuda")
    z_full, y_full = c.run(x)
    z, y = c.run(x, logits=False)
    assert z is None and torch.equal(y, y_full)
    z, y = c.run(x, labels=False)
    assert y is None and torch.equal(z, z_full)


def test_graph_capture_and_reprepare():
    from uaps_b200.unet import inference_params
    model = _model(3, 4, seed=3)
    c = CInfer(model, 3, 4)
    x = torch.randn(2, 3, 64, 64, device="cuda")
    z_eager, y_eager = c.run(x)
    out = (torch.empty_like(z_eager), torch.empty_like(y_eager))
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        c.run(x, out=out)                                 # warm-up off the capture
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        c.run(x, out=out)
    out[0].zero_()
    out[1].zero_()
    g.replay()
    assert torch.equal(out[0], z_eager) and torch.equal(out[1], y_eager)
    # new weights: a second prepare into the same state changes what the captured graph computes
    first = inference_params(model).clone()
    new = _model(3, 4, seed=4)
    model.load_state_dict(new.state_dict())
    c.prepare(inference_params(model))
    g.replay()
    want = model.predict(x)
    assert not torch.equal(want, z_eager)
    assert torch.equal(out[0], want) and torch.equal(out[1], _torch_labels(want))
    # prepare captured too: a graph that re-folds from a static blob, here back to the first weights
    blob = inference_params(model).clone()
    gp = torch.cuda.CUDAGraph()
    with torch.cuda.graph(gp):
        c.prepare(blob)
    blob.copy_(first)
    gp.replay()
    g.replay()
    assert torch.equal(out[0], z_eager) and torch.equal(out[1], y_eager)


def test_checkpoint_round_trip(tmp_path):
    from uaps_b200.unet import inference_params, save_checkpoint
    model = _model(1, 2, seed=6)
    opt = torch.optim.Adam(model.parameters(), lr=1e-3)
    path = str(tmp_path / "ck.pth")
    save_checkpoint(path, model, opt, epoch=3, best_dice=0.5)
    sd = torch.load(path, map_location="cuda")["state_dict"]
    assert all(k.startswith("module.") for k in sd)
    blob = inference_params(sd)
    assert torch.equal(blob, inference_params(model))
    c = CInfer(model, 1, 2)
    c.prepare(blob)
    x = torch.randn(2, 1, 128, 64, device="cuda")
    assert torch.equal(c.run(x)[0], model.predict(x))


def test_c_example_matches_predict(tmp_path):
    from uaps_b200.build import NVCC
    from uaps_b200.unet import inference_params
    libdir = os.path.join(ROOT, "uaps_b200", "lib")
    exe = str(tmp_path / "infer_c")
    r = subprocess.run([NVCC, "-O2", "-Wno-deprecated-gpu-targets", "-I", os.path.join(ROOT, "include"),
                        os.path.join(ROOT, "examples", "infer_c.c"), "-L", libdir, "-luaps_b200", "-Xlinker",
                        f"-rpath,{libdir}", "-o", exe], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    B, cin, H, W, C = 3, 3, 96, 128, 7
    model = _model(cin, C, seed=8)
    x = torch.randn(B, cin, H, W, device="cuda")
    inference_params(model).cpu().numpy().tofile(tmp_path / "params.bin")
    x.cpu().numpy().tofile(tmp_path / "x.bin")
    r = subprocess.run([exe, str(tmp_path / "params.bin"), str(cin), str(C), str(tmp_path / "x.bin"), str(B), str(H), str(W),
                        str(tmp_path / "logits.bin"), str(tmp_path / "labels.bin")], capture_output=True, text=True,
                       timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    want = model.predict(x).cpu()
    z = torch.from_numpy(np.fromfile(tmp_path / "logits.bin", dtype=np.float32).reshape(B, C, H, W))
    y = torch.from_numpy(np.fromfile(tmp_path / "labels.bin", dtype=np.uint8).reshape(B, H, W))
    assert torch.equal(z, want)
    assert torch.equal(y, _torch_labels(want))
