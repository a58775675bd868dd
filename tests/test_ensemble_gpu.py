"""Ensemble inference (DESIGN.md f5): the uaps_ensemble_head kernel against the oracle's mean prediction and KL maps
(oracle/uaps_loss_ref.py as torch CUDA ops), and UNet_UAPS.predict_uncertainty against the pieces it replaces."""
import numpy as np
import pytest
import torch

from oracle.uaps_loss_ref import unlabeled_loss_ref

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda:0")


def _oracle_head(logits):
    """q = preds (UAPS_train.py:223) and the mean KL map (1/K) sum_k var_k (:226-241) of the oracle, torch CUDA ops."""
    K = len(logits)
    ref = unlabeled_loss_ref(logits, [1.0 / K] * K, 0.0, 0.0)
    acc = ref["soft"][0]
    for k in range(1, K):
        acc = acc + ref["soft"][k]
    vsum = ref["var"][0]
    for k in range(1, K):
        vsum = vsum + ref["var"][k]
    return acc / K, vsum / K, acc


def _head(logits, **kw):
    from uaps_b200.ensemble import ensemble_uncertainty
    return ensemble_uncertainty(logits, **kw)


def _map_tol(ref):
    # 1e-5 of the map's largest value.  With K = 1 the oracle's map is pure rounding noise (log(softmax) - log_softmax,
    # ~1e-7) while the kernel's is 0: the floor of 0.1 in the scale keeps the bound at 1e-6 there.
    return 1e-5 * max(ref.abs().max().item(), 0.1)


@pytest.mark.parametrize("scale", [2.0, 16.0])                  # plain N(0, 2^2) logits and peaked ones (x8)
@pytest.mark.parametrize("shape", [(2, 16, 24), (1, 10, 13), (3, 7, 9)])   # HW % 4 == 0, HW % 2 == 0, odd HW
@pytest.mark.parametrize("C", [2, 3, 4, 7, 8])
@pytest.mark.parametrize("K", [1, 2, 3, 4, 5, 6])
def test_head_matches_oracle(K, C, shape, scale):
    B, H, W = shape
    g = torch.Generator(device=DEV).manual_seed(1000 * K + 10 * C + H)
    logits = [torch.randn(B, C, H, W, device=DEV, generator=g) * scale for _ in range(K)]
    q, unc, _ = _oracle_head(logits)
    out = _head(logits, return_probs=True)
    assert out.labels.dtype == torch.uint8 and out.labels.shape == (B, H, W)
    assert torch.equal(out.labels.long(), torch.argmax(q, 1))
    assert (out.uncertainty - unc).abs().max().item() <= _map_tol(unc)
    assert (out.mean_prob - q).abs().max().item() <= 1e-5 * q.abs().max().item()
    ref_img = unc.double().mean((1, 2))
    assert ((out.image_uncertainty.double() - ref_img).abs() <= 1e-5 * ref_img.abs() + 1e-7).all(), \
        (out.image_uncertainty, ref_img)


def test_head_without_optional_outputs():
    from uaps_b200 import _lib as L
    logits = [torch.randn(2, 4, 16, 16, device=DEV) for _ in range(3)]
    full = _head(logits)
    labels = torch.empty(2, 16, 16, dtype=torch.uint8, device=DEV)
    L.check(L.lib().uaps_ensemble_head(L.ptr_array(logits), 3, 2, 4, 256, labels.data_ptr(), None, None, None, None, 0,
                                       L.stream_ptr()), "uaps_ensemble_head")
    assert torch.equal(labels, full.labels) and full.mean_prob is None


def test_exact_ties_from_duplicated_class_planes():
    for K in (1, 2, 4):
        logits = []
        for _ in range(K):
            z = torch.randn(2, 5, 32, 32, device=DEV)
            z[:, 1] += 3.0
            z[:, 3] = z[:, 1]                                   # classes 1 and 3 tie exactly and lead
            z[:, 4] = z[:, 0]
            logits.append(z)
        q, _, _ = _oracle_head(logits)
        out = _head(logits)
        assert torch.equal(out.labels.long(), torch.argmax(q, 1))
        assert (out.labels == 1).float().mean().item() > 0.9 and not (out.labels == 3).any()


@pytest.mark.parametrize("K,gap", [(3, 1.5), (5, 10.0)])
def test_ties_decided_by_the_division_by_k(K, gap):
    """Three leading classes whose logits differ by at most two ulp: their summed probabilities differ in the last bits,
    and rounding the mean (acc / K) makes some of them equal -- torch's argmax of q then takes the lower index where the
    argmax of the sum would not.  That can only happen where 1/K shrinks the ulp spacing of the sum (acc in
    [0.75, 1) for K = 3, in [1.6, 2) for K = 5): `gap` (the 4th class's distance) puts the leading p_c there.  The test
    asserts that such pixels occur and that the kernel follows torch on all."""
    g = torch.Generator(device=DEV).manual_seed(K)
    logits = []
    for _ in range(K):
        lead = torch.rand(4, 128, 128, device=DEV, generator=g) + 3.0
        z = torch.empty(4, 4, 128, 128, device=DEV)
        for c in range(3):
            ulps = torch.randint(-2, 3, (4, 128, 128), device=DEV, generator=g).float() if c else 0.0
            z[:, c] = lead + ulps * torch.finfo(torch.float32).eps * 2.0      # lead in [3, 4): one ulp = 2 eps
        z[:, 3] = lead - gap
        logits.append(z)
    q, _, acc = _oracle_head(logits)
    decided = (torch.argmax(acc, 1) != torch.argmax(q, 1)).sum().item()
    assert decided > 0, "construction produced no tie that the division decides"
    out = _head(logits)
    assert torch.equal(out.labels.long(), torch.argmax(q, 1)), decided


def test_deterministic_and_argument_errors():
    g = torch.Generator(device=DEV).manual_seed(7)
    logits = [torch.randn(8, 4, 128, 128, device=DEV, generator=g) * 2 for _ in range(4)]
    a, b = _head(logits, return_probs=True), _head(logits, return_probs=True)
    for x, y in zip(a, b):
        assert torch.equal(x, y)
    z = logits[0]
    bad = [
        [z] * 7,                                                        # K > KMAX
        [torch.randn(1, 9, 8, 8, device=DEV)] * 2,                      # C > CMAX
        [torch.randn(1, 1, 8, 8, device=DEV)] * 2,                      # C < 2
        [z, z[:, :, :64]],                                              # shape mismatch
        [z.cpu(), z.cpu()],                                             # CPU tensors
        [z.double(), z.double()],                                       # not fp32
        [z[0], z[0]],                                                   # not 4-d
    ]
    for case in bad:
        with pytest.raises(RuntimeError):
            _head(case)


# ---- model level -------------------------------------------------------------------------------------------------
def _eval_model(n_aux, C, seed):
    from uaps_b200.unet import UNet_UAPS
    torch.manual_seed(seed)
    m = UNet_UAPS(3, C, n_aux=n_aux, compute="bf16").to(DEV)
    with torch.no_grad():                                   # non-trivial running statistics and affine parameters
        for mod in m.modules():
            if isinstance(mod, torch.nn.BatchNorm2d):
                mod.running_mean.normal_(0, 0.2); mod.running_var.uniform_(0.5, 1.5)
                mod.weight.uniform_(0.7, 1.3); mod.bias.normal_(0, 0.1)
    return m.eval()


def _draws(seed, n_aux):
    """The (key, u) pairs predict_uncertainty derives from an int seed, re-derived from its docstring."""
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(5 * (1 + max(0, n_aux - 3))):
        key = int(rng.integers(0, 2 ** 63 - 1))
        out.append((key, float(rng.uniform(0.7, 0.9))))
    return out


@torch.no_grad()
def _reference_logits(m, x, seed):
    """The same ensemble from existing pieces: unfolded eval-mode encoder (_encode16), explicit perturb3_nhwc per level
    with the seed-derived draws, unfolded decoders (_decode16)."""
    from uaps_b200.perturb import perturb3_nhwc
    from uaps_b200.unet import _AUX_KINDS
    d = _draws(seed, m.n_aux)
    feats = m._encode16(x, None)
    live = tuple(a <= m.n_aux for a in (1, 2, 3))
    per = [perturb3_nhwc(f, seed=d[l][0], u=d[l][1], outputs=live) for l, f in enumerate(feats)]
    logits = [m._decode16(feats, m.main_decoder)]
    for a in range(1, m.n_aux + 1):
        kind = _AUX_KINDS[(a - 1) % 3]
        if a <= 3:
            pf = [t[a - 1] for t in per]
        else:
            sel = tuple(k == kind for k in _AUX_KINDS)
            pf = [perturb3_nhwc(f, seed=d[5 * (a - 3) + l][0], u=d[5 * (a - 3) + l][1], outputs=sel)[_AUX_KINDS.index(kind)]
                  for l, f in enumerate(feats)]
        logits.append(m._decode16(pf, m.get_submodule(f"aux_decoder{a}")))
    return logits


@pytest.mark.parametrize("n_aux,C,shape", [(3, 4, (4, 3, 64, 96)), (4, 2, (2, 3, 240, 640))])
def test_predict_uncertainty_matches_the_pieces_it_replaces(n_aux, C, shape):
    m = _eval_model(n_aux, C, seed=3)
    x = torch.randn(*shape, device=DEV)
    got = m.predict_uncertainty(x, seed=21, return_probs=True)
    q, unc, _ = _oracle_head(_reference_logits(m, x, 21))
    B, _, H, W = shape
    assert got.labels.shape == (B, H, W) and got.uncertainty.shape == (B, H, W) and got.image_uncertainty.shape == (B,)
    rel_q = ((got.mean_prob - q).norm() / q.norm()).item()
    agree = (got.labels.long() == torch.argmax(q, 1)).float().mean().item()
    rel_u = ((got.uncertainty - unc).norm() / unc.norm()).item()
    rel_img = ((got.image_uncertainty - unc.mean((1, 2))).abs() / unc.mean((1, 2))).max().item()
    print(f"n_aux={n_aux} C={C} {shape}: mean_prob rel {rel_q:.3e}  labels agree {agree:.4f}  "
          f"uncertainty rel {rel_u:.3e}  image_uncertainty rel {rel_img:.3e}")
    assert rel_q < 2e-2, rel_q
    assert agree > 0.97, agree
    # The folded path (BatchNorm folded into bf16 weights, LeakyReLU in the epilogue) and the unfolded one differ by bf16
    # roundings in every layer of every decoder.  The uncertainty map is a difference of K such decoders' log-probabilities,
    # so its relative error is about 15x that of mean_prob: measured on B200, 1.7e-3 (map, both shapes) and 1.1e-3 /
    # 4.0e-4 (per-image means) against 1.2e-4 / 0.9e-4 for mean_prob.  The bounds leave ~6x headroom over that.
    assert rel_u < 1e-2, rel_u
    assert rel_img < 6e-3, rel_img


def test_predict_unchanged_and_aux_plan_lazy():
    m = _eval_model(3, 4, seed=4)
    x = torch.randn(2, 3, 64, 64, device=DEV)
    before = m.predict(x).clone()
    assert len(m._infer_plan[3]) == 0                      # predict packs no auxiliary decoder
    m.predict_uncertainty(x, seed=1)
    assert sorted(m._infer_plan[3]) == [1, 2, 3]
    assert torch.equal(m.predict(x), before)


def test_seeds_and_clean_main_decoder():
    m = _eval_model(1, 4, seed=5)
    x = torch.randn(2, 3, 64, 64, device=DEV)
    a, b = m.predict_uncertainty(x, seed=8, return_probs=True), m.predict_uncertainty(x, seed=8, return_probs=True)
    for u, v in zip(a, b):
        assert torch.equal(u, v)
    c = m.predict_uncertainty(x, seed=9, return_probs=True)
    assert not torch.equal(a.uncertainty, c.uncertainty)
    main = torch.softmax(m.predict(x), 1)
    for seed, out in ((8, a), (9, c)):
        draws = torch.from_numpy(m._ensemble_draws(seed)).to(DEV)
        logits = m._ensemble_logits16(x, draws)
        assert torch.equal(logits[0], m.predict(x))                    # the main decoder sees the clean features
        aux = 2 * out.mean_prob - main                                  # K * q - softmax(main) = softmax(aux)
        assert (aux - torch.softmax(logits[1], 1)).abs().max().item() <= 1e-5
    assert not torch.equal(2 * a.mean_prob - main, 2 * c.mean_prob - main)
    assert torch.equal(torch.softmax(m.predict(x), 1), main)


def test_graphed_replay():
    m = _eval_model(3, 4, seed=6)
    for B in (1, 3):
        x1, x2 = torch.randn(B, 3, 64, 64, device=DEV), torch.randn(B, 3, 64, 64, device=DEV)
        e1, e2 = m.predict_uncertainty(x1, seed=11), m.predict_uncertainty(x2, seed=12)
        g1 = [t.clone() for t in m.predict_uncertainty_graphed(x1, seed=11)[:3]]
        g2 = [t.clone() for t in m.predict_uncertainty_graphed(x2, seed=12)[:3]]     # pure replay: new input, new draws
        for e, g in ((e1, g1), (e2, g2)):
            for u, v in zip(e[:3], g):
                assert torch.equal(u, v)
        g3 = m.predict_uncertainty_graphed(x1, seed=13)
        assert not torch.equal(g3.uncertainty, g1[1])
    assert len([k for k in m._graphs if k[0] == "uncertainty"]) == 2
    m.train()
    assert "_graphs" not in m.__dict__ and m._infer_plan is None
    m.eval()
    m.predict_uncertainty_graphed(torch.randn(1, 3, 64, 64, device=DEV), seed=1)
    m.load_state_dict(m.state_dict())
    assert "_graphs" not in m.__dict__ and m._infer_plan is None


def test_fallback_paths():
    from uaps_b200.unet import UNet_UAPS
    x = torch.randn(2, 3, 32, 32, device=DEV)
    for m in (UNet_UAPS(3, 4, n_aux=2, compute="fp32").to(DEV).eval(), UNet_UAPS(3, 4, n_aux=2).to(DEV).train()):
        out = m.predict_uncertainty(x, return_probs=True)
        assert out.labels.shape == (2, 32, 32) and out.mean_prob.shape == (2, 4, 32, 32)
        assert torch.isfinite(out.uncertainty).all() and (out.uncertainty >= -1e-6).all()
