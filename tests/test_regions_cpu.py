"""Host side of the defect regions (no GPU needed): exports, the workspace size query, every argument check of
``uaps_regions`` (all of them come before any launch, so fake device addresses are never dereferenced), and the
numpy / scipy oracle against a plain-Python flood fill."""
import ctypes
from collections import deque

import numpy as np
import pytest

NEW = ("uaps_regions_workspace_bytes", "uaps_regions")


def test_exports():
    from uaps_b200 import _lib as L
    handle = ctypes.CDLL(L.LIB_PATH)
    for name in NEW:
        assert hasattr(handle, name) and name in L.exported_symbols()


def test_workspace_bytes():
    from uaps_b200 import _lib as L
    lib = L.lib()
    chunk = 2048
    for B, H, W, R in ((1, 1, 1, 0), (4, 17, 33, 5), (64, 256, 256, 256), (32, 240, 640, 0), (1, 1, 2**31 - 1, 1)):
        n = lib.uaps_regions_workspace_bytes(B, H, W, R)
        roots = -(-(B * -(-(H * W) // chunk) * 4) // 256) * 256          # int32 root count per pixel chunk, 256-aligned
        assert n == roots + 8 * B * R, (B, H, W, R)
    assert lib.uaps_regions_workspace_bytes(2, 64, 64, 300) > lib.uaps_regions_workspace_bytes(2, 64, 64, 0)
    for B, H, W, R in ((0, 8, 8, 1), (1, 0, 8, 1), (1, 8, -1, 1), (1, 8, 8, -1), (65536, 8, 8, 1), (1, 65536, 32768, 1)):
        assert lib.uaps_regions_workspace_bytes(B, H, W, R) == 0, (B, H, W, R)


def test_argument_checks():
    from uaps_b200 import _lib as L
    lib = L.lib()
    fake, odd, odd4 = (ctypes.c_void_p(a) for a in (4096, 4097, 4100))     # never dereferenced
    wb = lib.uaps_regions_workspace_bytes(2, 64, 64, 16)

    def run(labels=fake, unc=fake, B=2, H=64, W=64, regions=fake, count=fake, stats=fake, R=16, ws=fake, wbytes=wb):
        return lib.uaps_regions(labels, unc, B, H, W, regions, count, stats, R, ws, wbytes, None)

    for kw in ({"labels": None}, {"regions": None}, {"count": None}, {"ws": None}):
        assert run(**kw) == -1, kw
    assert run(stats=None) == -1                                     # stats needed when max_regions > 0
    assert run(R=0, wbytes=lib.uaps_regions_workspace_bytes(2, 64, 64, 0)) == -1   # ... and not passed otherwise
    for kw in ({"B": 0}, {"H": 0}, {"W": 0}, {"B": -1}, {"H": -3}, {"W": -64}, {"R": -1}):
        assert run(**kw) == -1, kw
    assert run(H=65536, W=32768) == -2 and run(H=1 << 16, W=1 << 15) == -2 and run(B=65536) == -2
    for kw in ({"unc": odd}, {"regions": odd}, {"count": odd}, {"stats": odd}, {"ws": odd4}):
        assert run(**kw) == -3, kw
    assert run(labels=odd, unc=None, regions=odd) == -3              # labels are bytes; any address is fine for them
    assert run(wbytes=wb - 1) == -1
    assert run(wbytes=lib.uaps_regions_workspace_bytes(1, 64, 64, 16)) == -1       # sized for a smaller batch
    # order: null pointers, then sizes, then range, then alignment, then the workspace size
    assert run(labels=None, B=0) == -1 and run(B=65536, regions=odd) == -2 and run(regions=odd, wbytes=0) == -3


def _flood_fill(labels):
    """Plain BFS over 8-neighbours of the same nonzero class, seeds visited in raster order: canonical ids."""
    H, W = labels.shape
    out = np.zeros((H, W), dtype=np.int32)
    n = 0
    for y in range(H):
        for x in range(W):
            c = labels[y, x]
            if c == 0 or out[y, x]:
                continue
            n += 1
            out[y, x] = n
            q = deque([(y, x)])
            while q:
                cy, cx = q.popleft()
                for dy in (-1, 0, 1):
                    for dx in (-1, 0, 1):
                        ny, nx = cy + dy, cx + dx
                        if 0 <= ny < H and 0 <= nx < W and not out[ny, nx] and labels[ny, nx] == c:
                            out[ny, nx] = n
                            q.append((ny, nx))
    return out, n


@pytest.mark.parametrize("seed", range(6))
@pytest.mark.parametrize("density,classes", [(0.1, 1), (0.45, 3), (0.7, 7), (1.0, 4)])
def test_oracle_matches_flood_fill(seed, density, classes):
    from oracle.regions_ref import regions_ref_image
    rng = np.random.default_rng(seed * 100 + classes)
    H, W = rng.integers(1, 24, size=2)
    fg = rng.random((H, W)) < density
    labels = np.where(fg, rng.integers(1, classes + 1, size=(H, W)), 0).astype(np.uint8)
    unc = rng.random((H, W)).astype(np.float32)
    want, n = _flood_fill(labels)
    got = regions_ref_image(labels, unc)
    assert got["count"] == n
    np.testing.assert_array_equal(got["regions"], want)
    for i in range(n):
        ys, xs = np.nonzero(want == i + 1)
        assert got["area"][i] == ys.size
        assert tuple(got["bbox"][i]) == (ys.min(), xs.min(), ys.max() + 1, xs.max() + 1)
        assert got["cls"][i] == labels[ys[0], xs[0]]
        assert got["unc_mean"][i] == np.float32(unc[ys, xs].astype(np.float64).sum() / ys.size)
    assert regions_ref_image(labels)["unc_mean"].tolist() == [0.0] * n


def test_oracle_keeps_diagonal_neighbours_of_different_classes_apart():
    from oracle.regions_ref import regions_ref_image
    labels = np.array([[1, 2, 1, 2],
                       [2, 1, 2, 1],
                       [1, 2, 1, 2]], dtype=np.uint8)      # two interleaved diagonal classes: 8-connected each
    got = regions_ref_image(labels)
    assert got["count"] == 2
    np.testing.assert_array_equal(got["regions"], np.where(labels == 1, 1, 2))
    assert got["cls"].tolist() == [1, 2] and got["area"].tolist() == [6, 6]
    side = np.array([[1, 2], [2, 1]], dtype=np.uint8)       # an 8-neighbour of another class is a different region
    assert regions_ref_image(side)["count"] == 2
    assert regions_ref_image(np.zeros((3, 5), np.uint8))["count"] == 0
