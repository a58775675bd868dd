"""Ensemble uncertainty inference through the C ABI on the B200: uaps_unet_ensemble_prepare folds and packs every
decoder exactly as UNet_UAPS._fold_bn / PackedConv do, uaps_unet_ensemble_run returns predict_uncertainty's labels,
uncertainty maps and mean prediction bit for bit from the same draws, inside a CUDA graph too, and
examples/uncertainty_c.c does the same with no Python."""
import ctypes
import os
import subprocess

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _model(cin, C, n_aux, seed=0):
    """Eval-mode model whose BatchNorms carry non-trivial running statistics and affine parameters."""
    from uaps_b200.unet import UNet_UAPS
    torch.manual_seed(seed)
    model = UNet_UAPS(cin, C, n_aux=n_aux).cuda().eval()
    with torch.no_grad():
        for m in model.modules():
            if isinstance(m, torch.nn.BatchNorm2d):
                m.running_mean.normal_(0, 0.1)
                m.running_var.uniform_(0.5, 1.5)
                m.weight.normal_(1, 0.1)
                m.bias.normal_(0, 0.1)
    return model


def _draws(model, seed):
    return torch.from_numpy(model._ensemble_draws(seed)).cuda()


class CEnsemble:
    """prepare + run over the raw entry points, on torch's current stream."""

    def __init__(self, model, cin, C, n_aux):
        from uaps_b200 import _lib as L
        from uaps_b200.unet import inference_params
        self.L, self.lib, self.cin, self.C, self.n_aux = L, L.lib(), cin, C, n_aux
        self.state = torch.empty(self.lib.uaps_unet_ensemble_state_bytes(cin, C, n_aux), dtype=torch.uint8, device="cuda")
        self.prepare(inference_params(model, ensemble=True))

    def prepare(self, blob):
        self.L.check(self.lib.uaps_unet_ensemble_prepare(blob.data_ptr(), self.cin, self.C, self.n_aux,
                                                         self.state.data_ptr(), self.state.numel(), self.L.stream_ptr()),
                     "prepare")

    def outputs(self, B, H, W, which=(True, True, True, True)):
        shapes = ((B, H, W), (B, H, W), (B,), (B, self.C, H, W))
        dtypes = (torch.uint8, torch.float32, torch.float32, torch.float32)
        return [torch.empty(s, dtype=d, device="cuda") if w else None for s, d, w in zip(shapes, dtypes, which)]

    def run(self, x, draws, out=None, ws=None):
        B, _, H, W = x.shape
        if ws is None:
            ws = torch.empty(self.lib.uaps_unet_ensemble_workspace_bytes(self.cin, self.C, self.n_aux, B, H, W),
                             dtype=torch.uint8, device="cuda")
        out = self.outputs(B, H, W) if out is None else out
        ptr = [None if t is None else t.data_ptr() for t in out]
        self.L.check(self.lib.uaps_unet_ensemble_run(self.state.data_ptr(), self.state.numel(), self.cin, self.C,
                                                     self.n_aux, x.data_ptr(), B, H, W, draws.data_ptr(), ws.data_ptr(),
                                                     ws.numel(), *ptr, self.L.stream_ptr()), "run")
        self.ws = ws
        return out


def _assert_equal(got, want):
    for name, g, w in zip(("labels", "uncertainty", "image_uncertainty", "mean_prob"), got, want):
        if g is not None:
            assert torch.equal(g, w), name


@pytest.mark.parametrize("n_aux", [1, 3, 5])
def test_prepare_folds_and_packs_like_the_python_plan(n_aux):
    from uaps_b200.conv import PackedConv
    from uaps_b200.unet import inference_params
    model = _model(3, 4, n_aux)
    c = CEnsemble(model, 3, 4, n_aux)
    # the packer writes only the bytes the selected kernel reads: both packings go into zero-filled buffers
    c.state.zero_()
    c.prepare(inference_params(model, ensemble=True))
    torch.cuda.synchronize()
    make = lambda w, b, cin_split=None: (w, b, cin_split)       # noqa: E731
    enc, dec, out = model._main_plan(make=make)
    layers = [l for blk in enc for l in blk] + [l for lvl in dec for l in lvl] + [out]
    plans = [None] * len(layers)
    for a in range(1, n_aux + 1):
        adec, aout = model._decoder_plan(model.get_submodule(f"aux_decoder{a}"), make=make)
        layers += [l for lvl in adec for l in lvl] + [aout]
        pdec, pout = model._aux_plan(a)                         # the PackedConvs predict_uncertainty runs
        plans += [p for lvl in pdec for p in lvl] + [pout]
    assert len(layers) == 23 + 13 * n_aux
    state = c.state.cpu()
    o = [ctypes.c_size_t() for _ in range(4)]
    for i, ((w, b, split), pc) in enumerate(zip(layers, plans)):
        assert c.lib.uaps_unet_ensemble_layer(3, 4, n_aux, i, *[ctypes.byref(v) for v in o]) == 0
        w_off, b_off, p_off, p_n = (v.value for v in o)
        got_w = state[w_off:w_off + 4 * w.numel()].view(torch.float32).view_as(w)
        got_b = state[b_off:b_off + 4 * b.numel()].view(torch.float32)
        assert torch.equal(got_w, w.float().cpu()), f"layer {i} weight"
        assert torch.equal(got_b, b.float().cpu()), f"layer {i} bias"
        if pc is None:
            pc = PackedConv(w, b, cin_split=split)
        else:
            assert torch.equal(pc.bias.cpu(), got_b), f"layer {i} plan bias"
        pc.packed.zero_()
        pc._pack(w.detach().float().contiguous())
        packed = pc.packed.cpu()
        assert p_n == packed.numel() and torch.equal(state[p_off:p_off + p_n], packed), f"layer {i} packed"


CASES = [((4, 3, 64, 96), 4, 3), ((2, 3, 240, 640), 2, 4), ((1, 1, 512, 512), 2, 3), ((2, 3, 64, 64), 7, 1),
         ((2, 3, 64, 64), 3, 5), ((1, 3, 256, 256), 4, 3)]


@pytest.mark.parametrize("shape,C,n_aux", CASES)
def test_run_equals_predict_uncertainty(shape, C, n_aux):
    B, cin, H, W = shape
    seed = 11 + B + C + n_aux
    model = _model(cin, C, n_aux, seed=B + C)
    c = CEnsemble(model, cin, C, n_aux)
    x = torch.randn(*shape, device="cuda", generator=torch.Generator(device="cuda").manual_seed(7))
    got = c.run(x, _draws(model, seed))
    want = model.predict_uncertainty(x, seed=seed, return_probs=True)
    _assert_equal(got, want)
    assert want.uncertainty.abs().sum() > 0                    # the decoders disagree somewhere: the maps are not trivial


def test_optional_outputs():
    model = _model(3, 4, 3, seed=2)
    c = CEnsemble(model, 3, 4, 3)
    x = torch.randn(2, 3, 64, 128, device="cuda")
    d = _draws(model, 5)
    full = c.run(x, d)
    for which in ((True, False, False, False), (True, False, True, True), (True, True, False, True),
                  (True, True, True, False)):
        got = c.run(x, d, out=c.outputs(2, 64, 128, which))
        assert all((g is None) == (not w) for g, w in zip(got, which))
        _assert_equal(got, full)


def test_graph_capture_new_draws_and_reprepare():
    from uaps_b200.unet import inference_params
    model = _model(3, 4, 4, seed=3)
    c = CEnsemble(model, 3, 4, 4)
    x = torch.randn(2, 3, 64, 64, device="cuda")
    x_static, d_static = x.clone(), _draws(model, 1)
    eager = [t.clone() for t in c.run(x_static, d_static)]
    out = c.outputs(2, 64, 64)
    ws = torch.empty_like(c.ws)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        c.run(x_static, d_static, out=out, ws=ws)              # warm-up off the capture
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        c.run(x_static, d_static, out=out, ws=ws)
    for t in out:
        t.zero_()
    g.replay()
    _assert_equal(out, eager)
    # a new input and new draws written into the captured buffers
    x2 = torch.randn(2, 3, 64, 64, device="cuda")
    x_static.copy_(x2)
    d_static.copy_(_draws(model, 2))
    g.replay()
    _assert_equal(out, model.predict_uncertainty(x2, seed=2, return_probs=True))
    _assert_equal(c.run(x2, _draws(model, 2)), out)
    # new weights: a second prepare into the same state changes what the captured graph computes
    model.load_state_dict(_model(3, 4, 4, seed=4).state_dict())
    c.prepare(inference_params(model, ensemble=True))
    g.replay()
    want = model.predict_uncertainty(x2, seed=2, return_probs=True)
    assert not torch.equal(want.mean_prob, eager[3])
    _assert_equal(out, want)


def test_deterministic():
    model = _model(3, 2, 5, seed=9)
    c = CEnsemble(model, 3, 2, 5)
    x = torch.randn(3, 3, 96, 128, device="cuda")
    d = _draws(model, 3)
    first = [t.clone() for t in c.run(x, d)]
    _assert_equal(c.run(x, d), first)


def test_checkpoint_round_trip(tmp_path):
    from uaps_b200.unet import inference_params, save_checkpoint
    model = _model(1, 2, 3, seed=6)
    opt = torch.optim.Adam(model.parameters(), lr=1e-3)
    path = str(tmp_path / "ck.pth")
    save_checkpoint(path, model, opt, epoch=3, best_dice=0.5)
    sd = torch.load(path, map_location="cuda")["state_dict"]
    assert all(k.startswith("module.") for k in sd)
    blob = inference_params(sd, ensemble=True)
    assert torch.equal(blob, inference_params(model, ensemble=True))
    c = CEnsemble(model, 1, 2, 3)
    c.prepare(blob)
    x = torch.randn(2, 1, 128, 64, device="cuda")
    _assert_equal(c.run(x, _draws(model, 4)), model.predict_uncertainty(x, seed=4, return_probs=True))


def test_c_example_matches_predict_uncertainty(tmp_path):
    from uaps_b200.build import NVCC
    from uaps_b200.unet import inference_params
    libdir = os.path.join(ROOT, "uaps_b200", "lib")
    exe = str(tmp_path / "uncertainty_c")
    r = subprocess.run([NVCC, "-O2", "-Wno-deprecated-gpu-targets", "-I", os.path.join(ROOT, "include"),
                        os.path.join(ROOT, "examples", "uncertainty_c.c"), "-L", libdir, "-luaps_b200", "-Xlinker",
                        f"-rpath,{libdir}", "-o", exe], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    B, cin, H, W, C, n_aux, seed = 3, 3, 96, 128, 7, 4, 21
    model = _model(cin, C, n_aux, seed=8)
    x = torch.randn(B, cin, H, W, device="cuda")
    inference_params(model, ensemble=True).cpu().numpy().tofile(tmp_path / "params.bin")
    x.cpu().numpy().tofile(tmp_path / "x.bin")
    model._ensemble_draws(seed).tofile(tmp_path / "draws.bin")
    files = [str(tmp_path / n) for n in ("labels.bin", "unc.bin", "img.bin")]
    r = subprocess.run([exe, str(tmp_path / "params.bin"), str(cin), str(C), str(n_aux), str(tmp_path / "x.bin"),
                        str(tmp_path / "draws.bin"), str(B), str(H), str(W), *files], capture_output=True, text=True,
                       timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    want = model.predict_uncertainty(x, seed=seed)
    got = (torch.from_numpy(np.fromfile(files[0], dtype=np.uint8).reshape(B, H, W)),
           torch.from_numpy(np.fromfile(files[1], dtype=np.float32).reshape(B, H, W)),
           torch.from_numpy(np.fromfile(files[2], dtype=np.float32).reshape(B)))
    for name, g, w in zip(("labels", "uncertainty", "image_uncertainty"), got, want):
        assert torch.equal(g, w.cpu()), name
