"""The float64 SSIM reference (tests/ssim_reference.py) against independent formulations, and the SSIM C-ABI without a GPU."""
import numpy as np
import pytest
import torch

from dt4image_restoration_b200 import _lib
from ssim_reference import gaussian_window, ssim

SHAPES = [(11, 11), (16, 16), (45, 51), (130, 136)]


def _pair(H, W, seed, n=2):
    g = torch.Generator().manual_seed(seed)
    x = torch.rand(n, 1, H, W, generator=g, dtype=torch.float64) * 1.4 - 0.2
    y = torch.rand(n, 1, H, W, generator=g, dtype=torch.float64)
    return x, y


def _ssim_scipy(x, y):
    """Same definition through scipy.ndimage.gaussian_filter (radius int(3.5 * 1.5 + 0.5) = 5), cropped to the valid map."""
    from scipy.ndimage import gaussian_filter
    X = np.clip(x, 0, 1)

    def f(a):
        return gaussian_filter(a, 1.5, truncate=3.5)[5:-5, 5:-5]

    mx, my = f(X), f(y)
    sxx, syy, sxy = f(X * X) - mx * mx, f(y * y) - my * my, f(X * y) - mx * my
    c1, c2 = 0.01 ** 2, 0.03 ** 2
    return float((((2 * mx * my + c1) * (2 * sxy + c2)) / ((mx * mx + my * my + c1) * (sxx + syy + c2))).mean())


def _ssim_direct(x, y):
    """Non-separable: the 11x11 window g (x) g summed directly at every valid position."""
    g = gaussian_window().numpy()
    w2 = np.outer(g, g)
    X = np.clip(x, 0, 1)
    H, W = X.shape
    vals = []
    for i in range(H - 10):
        for j in range(W - 10):
            a, b = X[i:i + 11, j:j + 11], y[i:i + 11, j:j + 11]
            mx, my = (w2 * a).sum(), (w2 * b).sum()
            sxx = (w2 * a * a).sum() - mx * mx
            syy = (w2 * b * b).sum() - my * my
            sxy = (w2 * a * b).sum() - mx * my
            c1, c2 = 0.01 ** 2, 0.03 ** 2
            vals.append(((2 * mx * my + c1) * (2 * sxy + c2)) / ((mx * mx + my * my + c1) * (sxx + syy + c2)))
    return float(np.mean(vals))


@pytest.mark.parametrize("H,W", SHAPES)
def test_reference_matches_scipy_gaussian_filter(H, W):
    x, y = _pair(H, W, seed=H * 1000 + W)
    ref = ssim(x, y)
    assert ref.shape == (2, 1) and ref.dtype == torch.float64
    for b in range(2):
        assert abs(float(ref[b, 0]) - _ssim_scipy(x[b, 0].numpy(), y[b, 0].numpy())) <= 1e-12


@pytest.mark.parametrize("H,W", [(11, 11), (20, 17)])
def test_reference_matches_direct_window_sum(H, W):
    x, y = _pair(H, W, seed=7 + H + W)
    ref = ssim(x, y)
    for b in range(2):
        assert abs(float(ref[b, 0]) - _ssim_direct(x[b, 0].numpy(), y[b, 0].numpy())) <= 1e-12


def test_identical_images_give_one():
    _, y = _pair(45, 51, seed=3)
    assert torch.allclose(ssim(y, y), torch.ones(2, 1, dtype=torch.float64), rtol=0, atol=1e-12)


def test_constant_pair_gives_one():
    x = torch.full((1, 1, 32, 40), 0.3, dtype=torch.float64)
    assert abs(float(ssim(x, x.clone())[0, 0]) - 1.0) <= 1e-12


def test_output_is_clamped_gt_is_not():
    x, y = _pair(30, 33, seed=11)
    assert float(x.min()) < 0 and float(x.max()) > 1
    assert torch.equal(ssim(x, y), ssim(x.clamp(0, 1), y))
    assert not torch.equal(ssim(y, x), ssim(y, x.clamp(0, 1)))


def test_shared_gt_broadcasts():
    x, y = _pair(24, 24, seed=5, n=3)
    shared = ssim(x, y[0, 0])
    for b in range(3):
        assert torch.equal(shared[b], ssim(x[b:b + 1], y[0:1])[0])


def test_workspace_bytes_without_gpu():
    lib = _lib.load()
    # 64 x 28 output tiles, one fp32 partial each, rounded up to 16 bytes
    assert lib.pnp_ssim_workspace_bytes(64, 256, 256) == 64 * 4 * 9 * 4
    assert lib.pnp_ssim_workspace_bytes(1, 11, 11) == 16
    assert lib.pnp_ssim_workspace_bytes(3, 2000, 37) == 3 * 72 * 4
    assert lib.pnp_ssim_workspace_bytes(1, 2000, 37) == 288
    for B, H, W in ((0, 64, 64), (1, 10, 64), (1, 64, 10)):
        assert lib.pnp_ssim_workspace_bytes(B, H, W) == 0


def test_ssim_fails_loudly_before_init():
    lib = _lib.load()
    if _lib._inited:
        pytest.skip("the library was already initialised in this process")
    rc = lib.pnp_ssim(None, None, 0, None, None, 1, 16, 16, None)
    assert rc == -3 and b"pnp_init" in lib.pnp_last_error()
