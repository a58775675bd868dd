"""Defect regions on the device (uaps_regions / uaps_b200.regions.defect_regions) against the numpy / scipy oracle.

Integer outputs (region map, counts, class, area, box) must be equal; unc_mean within 1 fp32 ulp of the oracle's fp64 mean
rounded to fp32 (fp64 atomics re-associate the sum).  Every call goes into outputs and a workspace pre-filled with 0xFF,
and the stats rows past the count must come back zero.  Map families: random multi-class noise from sparse to
percolating to full, smooth blobs, and shapes aimed at the merge across 32x32 tiles (serpentine, spiral, checkerboard,
diagonal-only links, lines on tile borders, two diagonally interleaved classes)."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

FIELDS = 8


def _dev():
    return torch.device("cuda:0")


def _call(labels, unc=None, max_regions=256):
    """uaps_regions through ctypes into 0xFF-filled outputs and workspace."""
    from uaps_b200 import _lib as L
    lib = L.lib()
    B, H, W = labels.shape
    dev = labels.device
    regions = torch.full((B, H, W), -1, dtype=torch.int32, device=dev)
    count = torch.full((B,), -1, dtype=torch.int32, device=dev)
    stats = torch.full((B, max(max_regions, 1), FIELDS), -1, dtype=torch.int32, device=dev)
    nbytes = lib.uaps_regions_workspace_bytes(B, H, W, max_regions)
    ws = torch.full((nbytes,), 255, dtype=torch.uint8, device=dev)
    L.check(lib.uaps_regions(labels.data_ptr(), None if unc is None else unc.data_ptr(), B, H, W, regions.data_ptr(),
                             count.data_ptr(), stats.data_ptr() if max_regions > 0 else None, max_regions, ws.data_ptr(),
                             nbytes, L.stream_ptr()), "uaps_regions")
    torch.cuda.synchronize()
    return regions, count, stats[:, :max_regions]


def _compare(labels, unc, out, max_regions):
    from oracle.regions_ref import regions_ref
    regions, count, stats = (t.cpu().numpy() for t in out)
    refs = regions_ref(labels.cpu().numpy(), None if unc is None else unc.cpu().numpy())
    for b, ref in enumerate(refs):
        np.testing.assert_array_equal(regions[b], ref["regions"], err_msg=f"image {b}")
        assert count[b] == ref["count"], (b, count[b], ref["count"])
        k = min(ref["count"], max_regions)
        st = stats[b]
        np.testing.assert_array_equal(st[:k, 0], ref["cls"][:k])
        np.testing.assert_array_equal(st[:k, 1], ref["area"][:k])
        np.testing.assert_array_equal(st[:k, 2:6], ref["bbox"][:k])
        assert (st[:k, 7] == 0).all()
        got = st[:k, 6].view(np.float32)
        want = ref["unc_mean"][:k]
        if unc is None:
            assert (got == 0).all()
        else:
            ulp = np.spacing(np.abs(want)).astype(np.float32)
            bad = np.abs(got.astype(np.float64) - want.astype(np.float64)) > ulp
            assert not bad.any(), (b, np.nonzero(bad)[0][:5], got[bad][:5], want[bad][:5])
        assert (st[k:] == 0).all(), f"image {b}: rows past the count are not zero"
    return refs


def _check(labels_np, unc=True, max_regions=256, seed=0):
    labels = torch.from_numpy(np.ascontiguousarray(labels_np, dtype=np.uint8)).to(_dev())
    u = None
    if unc:
        g = torch.Generator(device=_dev()).manual_seed(seed)
        u = torch.rand(labels.shape, generator=g, device=_dev()) * 3
    out = _call(labels, u, max_regions)
    return out, _compare(labels, u, out, max_regions)


# ---- map generators ----------------------------------------------------------------------------------------------------
def random_map(shape, density, classes, seed):
    rng = np.random.default_rng(seed)
    fg = rng.random(shape) < density
    return np.where(fg, rng.integers(1, classes + 1, size=shape), 0).astype(np.uint8)


def blob_map(shape, classes, seed, sigma=6.0, thresh=0.9):
    from scipy import ndimage
    rng = np.random.default_rng(seed)
    out = np.zeros(shape, dtype=np.uint8)
    for b in range(shape[0]):
        for c in range(1, classes + 1):
            f = ndimage.gaussian_filter(rng.standard_normal(shape[1:]), sigma)
            out[b][f > thresh * f.std()] = c
    return out


def serpentine(H, W):
    m = np.zeros((H, W), dtype=np.uint8)
    m[0::2] = 1
    for y in range(1, H, 2):
        m[y, W - 1 if (y // 2) % 2 == 0 else 0] = 1
    return m


def spiral(n):
    """A one-pixel-wide path winding inwards, ring by ring, two pixels apart."""
    m = np.zeros((n, n), dtype=np.uint8)
    top, left, bottom, right = 0, 0, n - 1, n - 1
    while top <= bottom and left <= right:
        m[top, left:right + 1] = 1
        m[top:bottom + 1, right] = 1
        if top + 2 <= bottom:
            m[bottom, left:right + 1] = 1
        if left + 2 <= right and top + 2 <= bottom:
            m[top + 2:bottom + 1, left] = 1
        top += 2; left += 2; bottom -= 2; right -= 2
        if top <= bottom and left - 1 >= 0:
            m[top, left - 1] = 1
    return m


def checkerboard(H, W, cls=1):
    yy, xx = np.mgrid[0:H, 0:W]
    return np.where((yy + xx) % 2 == 0, cls, 0).astype(np.uint8)


def diagonal_lines(H, W):
    yy, xx = np.mgrid[0:H, 0:W]
    m = np.zeros((H, W), dtype=np.uint8)
    m[(xx - yy) % 7 == 0] = 1          # down-right diagonals: tile borders crossed diagonally only
    m[(xx + yy) % 11 == 0] = 2         # down-left diagonals: the up-right link
    return m


def border_lines(H, W):
    m = np.zeros((H, W), dtype=np.uint8)
    for k in range(31, max(H, W) + 1, 32):
        if k < H:
            m[k, :] = 1
        if k + 1 < H:
            m[k + 1, ::3] = 2
        if k < W:
            m[:, k] = 3
        if k + 1 < W:
            m[1::2, k + 1] = 4
    return m


def interleaved(H, W):
    yy, xx = np.mgrid[0:H, 0:W]
    return (1 + (yy + xx) % 2).astype(np.uint8)


# ---- cases -------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("classes", [1, 4, 7])
@pytest.mark.parametrize("density", [0.05, 0.4, 0.6, 1.0])
def test_random_maps(density, classes):
    _check(random_map((6, 100, 131), density, classes, seed=int(density * 100) + classes), max_regions=4096)


def test_blobs():
    _check(blob_map((8, 256, 256), 3, seed=5), max_regions=512)


@pytest.mark.parametrize("H,W", [(64, 64), (255, 257), (512, 512)])
def test_serpentine(H, W):
    (_, count, _), _ = _check(serpentine(H, W)[None], max_regions=4)
    assert count.item() == 1


def test_spiral():
    (_, count, stats), _ = _check(spiral(301)[None], max_regions=4)
    assert count.item() == 1 and tuple(stats[0, 0, 2:6].tolist()) == (0, 0, 301, 301)


@pytest.mark.parametrize("H,W", [(64, 64), (97, 130)])
def test_checkerboard_is_one_region(H, W):
    (_, count, _), _ = _check(checkerboard(H, W)[None])
    assert count.item() == 1


def test_diagonal_links_across_tiles():
    _check(diagonal_lines(200, 333)[None], max_regions=1024)


def test_lines_on_tile_borders():
    _check(border_lines(161, 190)[None], max_regions=1024)


def test_two_classes_interleaved_diagonally():
    (_, count, _), _ = _check(interleaved(130, 97)[None])
    assert count.item() == 2


@pytest.mark.parametrize("B,H,W", [(3, 1, 1), (2, 1, 1000), (2, 1000, 1), (4, 17, 33), (2, 255, 257), (2, 31, 31),
                                   (2, 32, 32), (2, 33, 33), (2, 31, 33), (2, 63, 65), (1, 1, 70000)])
def test_shapes(B, H, W):
    _check(random_map((B, H, W), 0.45, 3, seed=H * 7 + W), max_regions=max(1, H * W))


@pytest.mark.parametrize("B,H,W", [(64, 256, 256), (32, 512, 512), (32, 240, 640)])
def test_batch_shapes(B, H, W):
    labels = blob_map((B, H, W), 2, seed=B + H) if B == 64 else random_map((B, H, W), 0.4, 4, seed=W)
    _check(labels, max_regions=256)


def test_one_large_image():
    labels = random_map((1, 2048, 2048), 0.4, 2, seed=11)
    labels[0, 1024:] = serpentine(1024, 2048)
    _check(labels, max_regions=1000)


def test_all_background_and_all_one_class():
    (regions, count, stats), _ = _check(np.zeros((2, 70, 90)))
    assert (regions == 0).all() and (count == 0).all() and (stats == 0).all()
    (regions, count, stats), _ = _check(np.full((2, 300, 257), 3))
    assert (regions == 1).all() and (count == 1).all()
    assert stats[:, 0, :6].tolist() == [[3, 300 * 257, 0, 0, 300, 257]] * 2


@pytest.mark.parametrize("max_regions", [0, 1, 7])
def test_max_regions_below_count(max_regions):
    (_, count, stats), refs = _check(random_map((3, 64, 80), 0.2, 3, seed=3), max_regions=max_regions)
    assert all(r["count"] > max_regions for r in refs)
    assert stats.shape == (3, max_regions, FIELDS)


def test_uncertainty_null_and_given():
    labels = blob_map((4, 128, 128), 2, seed=9)
    (r0, c0, s0), _ = _check(labels, unc=False)
    (r1, c1, s1), _ = _check(labels, unc=True)
    assert torch.equal(r0, r1) and torch.equal(c0, c1) and torch.equal(s0[..., :6], s1[..., :6])


def test_two_runs_bitwise_equal():
    labels = torch.from_numpy(random_map((8, 256, 256), 0.4, 3, seed=2)).to(_dev())
    unc = torch.rand(labels.shape, device=_dev())
    a, b = _call(labels, unc), _call(labels, unc)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1]) and torch.equal(a[2][..., :6], b[2][..., :6])


def test_defect_regions_api():
    from uaps_b200.regions import defect_regions
    labels = torch.from_numpy(blob_map((3, 96, 160), 3, seed=4)).to(_dev())
    unc = torch.rand(labels.shape, device=_dev())
    r = defect_regions(labels, unc, max_regions=64)
    regions, count, stats = _call(labels, unc, 64)
    assert torch.equal(r.regions, regions) and torch.equal(r.count, count)
    assert torch.equal(r.cls, stats[..., 0]) and torch.equal(r.area, stats[..., 1]) and torch.equal(r.bbox, stats[..., 2:6])
    _compare(labels, unc, (r.regions, r.count, torch.cat([r.cls[..., None], r.area[..., None], r.bbox,
                                                          r.unc_mean.view(torch.int32)[..., None],
                                                          torch.zeros_like(r.cls)[..., None]], -1)), 64)
    assert r.unc_mean.dtype == torch.float32 and r.regions.dtype == torch.int32
    with pytest.raises(RuntimeError, match="uint8"):
        defect_regions(labels.long())
    r0 = defect_regions(labels, max_regions=0)
    assert torch.equal(r0.regions, regions) and r0.cls.shape == (3, 0)


def test_graph_capture_and_replay_with_new_labels():
    from uaps_b200 import _lib as L
    lib = L.lib()
    B, H, W, R = 4, 192, 200, 128
    dev = _dev()
    labels = torch.from_numpy(blob_map((B, H, W), 2, seed=1)).to(dev)
    unc = torch.rand((B, H, W), device=dev)
    regions = torch.full((B, H, W), -1, dtype=torch.int32, device=dev)
    count = torch.full((B,), -1, dtype=torch.int32, device=dev)
    stats = torch.full((B, R, FIELDS), -1, dtype=torch.int32, device=dev)
    nbytes = lib.uaps_regions_workspace_bytes(B, H, W, R)
    ws = torch.full((nbytes,), 255, dtype=torch.uint8, device=dev)

    def run():
        L.check(lib.uaps_regions(labels.data_ptr(), unc.data_ptr(), B, H, W, regions.data_ptr(), count.data_ptr(),
                                 stats.data_ptr(), R, ws.data_ptr(), nbytes, L.stream_ptr()), "uaps_regions")

    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        run()
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        run()
    for seed, maker in ((2, lambda: blob_map((B, H, W), 3, seed=2)), (3, lambda: random_map((B, H, W), 0.4, 2, seed=3)),
                        (4, lambda: random_map((B, H, W), 0.02, 1, seed=4))):
        labels.copy_(torch.from_numpy(maker()))
        unc.copy_(torch.rand((B, H, W), device=dev, generator=torch.Generator(device=dev).manual_seed(seed)))
        regions.fill_(-1)
        graph.replay()
        torch.cuda.synchronize()
        _compare(labels, unc, (regions, count, stats), R)


def test_end_to_end_predict_uncertainty():
    from uaps_b200.regions import defect_regions
    from uaps_b200.unet import UNet_UAPS
    torch.manual_seed(0)
    model = UNet_UAPS(3, 4).to(_dev()).eval()
    g = torch.Generator(device=_dev()).manual_seed(7)
    x = torch.randn(4, 3, 128, 160, generator=g, device=_dev())
    labels, unc = model.predict_uncertainty(x, seed=3)[:2]
    r = defect_regions(labels, unc)
    assert int(r.count.sum()) > 0
    regions, count, stats = _call(labels, unc, 256)
    _compare(labels, unc, (regions, count, stats), 256)
    assert torch.equal(r.regions, regions) and torch.equal(r.count, count)
