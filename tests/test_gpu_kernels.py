"""Parity of each CUDA kernel (through the C-ABI) against the CPU oracle.  Needs a B200."""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from dt4image_restoration_b200 import ops, synth
from dt4image_restoration_b200.noise import UNetDenoiser2D
from oracle import pnp_oracle as O

pytestmark = pytest.mark.gpu
DEV = "cuda"


def bf16r(t):
    return t.to(torch.bfloat16).to(torch.float32)


# ------------------------------------------------------------------------------------------------
# PSNR (env.py:120-125)
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("N,H,W", [(1, 128, 128), (5, 256, 256), (3, 40, 40), (2, 33, 17), (130, 64, 64)])
def test_psnr_matches_oracle(N, H, W):
    g = torch.Generator().manual_seed(N * 1000 + H)
    x = torch.rand(N, H, W, generator=g) * 1.4 - 0.2      # exercises the clamp
    gt = torch.rand(N, H, W, generator=g)
    ref = O.psnr(x, gt).reshape(-1)
    got = ops.psnr(x.to(DEV), gt.to(DEV)).cpu()
    assert (got - ref).abs().max() < 1e-3          # dB; fp32 reduction-order noise only
    shared = ops.psnr(x.to(DEV), gt[:1].to(DEV)).cpu()
    ref_s = O.psnr(x, gt[:1].expand(N, -1, -1)).reshape(-1)
    assert (shared - ref_s).abs().max() < 1e-3


def test_psnr_against_reference_golden(golden_dir):
    gd = np.load(os.path.join(golden_dir, "ref_fft_psnr.npz"))
    gen = torch.Generator().manual_seed(7)
    for (h, w) in ((32, 32), (64, 48), (128, 128), (30, 34)):   # replay the generator stream of make_golden
        torch.randn(2, 1, h, w, generator=gen); torch.randn(2, 1, h, w, generator=gen)
    a = torch.rand(3, 40, 40, generator=gen) * 1.4 - 0.2
    b = torch.rand(3, 40, 40, generator=gen)
    got = ops.psnr(a.to(DEV), b.to(DEV)).cpu().reshape(3, 1)
    np.testing.assert_allclose(got.numpy(), gd["psnr"], rtol=0, atol=1e-3)


# ------------------------------------------------------------------------------------------------
# centred FFT (transformations.py:6-19)
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("H,W", [(32, 32), (64, 64), (128, 128), (256, 256), (512, 512), (64, 256), (512, 32), (128, 64)])
@pytest.mark.parametrize("inverse", [False, True])
def test_fft2c_matches_oracle(H, W, inverse):
    g = torch.Generator().manual_seed(H * 7 + W)
    z = torch.complex(torch.randn(2, 1, H, W, generator=g), torch.randn(2, 1, H, W, generator=g))
    ref = O.centered_ifft2(z) if inverse else O.centered_fft2(z)
    got = ops.fft2c(z.to(DEV), inverse=inverse).cpu()
    scale = ref.abs().max().item()
    assert (got - ref).abs().max().item() < 2e-6 * scale * np.log2(H * W)


def test_fft2c_golden_and_roundtrip(golden_dir):
    gd = np.load(os.path.join(golden_dir, "ref_fft_psnr.npz"))
    gen = torch.Generator().manual_seed(7)
    for (h, w) in ((32, 32), (64, 48), (128, 128), (30, 34)):   # 64x48 and 30x34: the dense-DFT path (fftprox_any.cuh)
        zc = torch.complex(torch.randn(2, 1, h, w, generator=gen), torch.randn(2, 1, h, w, generator=gen))
        got = torch.view_as_real(ops.fft2c(zc.to(DEV)).cpu()).numpy()
        np.testing.assert_allclose(got, gd[f"fft_{h}x{w}"], rtol=0, atol=3e-5)
        goti = torch.view_as_real(ops.fft2c(zc.to(DEV), inverse=True).cpu()).numpy()
        np.testing.assert_allclose(goti, gd[f"ifft_{h}x{w}"], rtol=0, atol=3e-5)
        rt = ops.fft2c(ops.fft2c(zc.to(DEV)), inverse=True).cpu()
        assert (rt - zc).abs().max() < 2e-5


@pytest.mark.parametrize("B,H,W", [(3, 130, 130), (2, 136, 120), (2, 33, 47), (1, 45, 51), (2, 17, 1000), (1, 1024, 16),
                                   (2, 16, 16), (1, 2, 3), (1, 1024, 1024)])
@pytest.mark.parametrize("inverse", [False, True])
def test_fft2c_any_size_matches_oracle(B, H, W, inverse):
    """Sizes the radix kernels do not serve (not a power of two in 32..512) go through the dense-DFT path; odd sizes are
    where ifftshift and fftshift differ (transformations.py:6-19)."""
    g = torch.Generator().manual_seed(H * 7 + W)
    z = torch.complex(torch.randn(B, 1, H, W, generator=g), torch.randn(B, 1, H, W, generator=g))
    ref = O.centered_ifft2(z) if inverse else O.centered_fft2(z)
    got = ops.fft2c(z.to(DEV), inverse=inverse).cpu()
    scale = ref.abs().max().item()
    assert (got - ref).abs().max().item() < 4e-6 * scale * np.log2(H * W)
    rt = ops.fft2c(ops.fft2c(z.to(DEV), inverse=inverse), inverse=not inverse).cpu()
    assert (rt - z).abs().max().item() < 3e-5


def test_fft2c_any_size_more_images_than_one_grid_dimension():
    """More images than gridDim.y holds (65535): the dense-DFT launcher walks the batch in slices."""
    B, H, W = 70001, 3, 5
    g = torch.Generator().manual_seed(5)
    z = torch.complex(torch.randn(B, 1, H, W, generator=g), torch.randn(B, 1, H, W, generator=g))
    got = ops.fft2c(z.to(DEV)).cpu()
    ref = O.centered_fft2(z)
    assert (got - ref).abs().max().item() < 1e-5
    assert (got[-1] - ref[-1]).abs().max().item() < 1e-5 and (got[65535] - ref[65535]).abs().max().item() < 1e-5


def test_radix_passes_more_images_than_one_grid_dimension():
    """More images than gridDim.y holds (65535) at a radix size: the radix line passes walk the batch in slices too, and an
    image's result does not depend on the slice it lands in."""
    B, H, W = 65537, 32, 32
    g = torch.Generator(device=DEV).manual_seed(13)
    cz = lambda: torch.complex(torch.randn(B, 1, H, W, device=DEV, generator=g),
                               torch.randn(B, 1, H, W, device=DEV, generator=g))
    z = cz()
    got = ops.fft2c(z)
    for b in (0, 65536):
        assert torch.equal(got[b], ops.fft2c(z[b:b + 1])[0])
    del got
    x = torch.rand(B, 1, H, W, device=DEV, generator=g)
    u, y0 = z, cz()
    mask = torch.rand(B, 1, H, W, device=DEV, generator=g) < 0.3
    mu = torch.tensor([0.4], device=DEV)
    zz, uu, vv = ops.prox_dual(x, u, y0, mask, mu)
    for b in (0, 65536):
        s = slice(b, b + 1)
        z1, u1, v1 = ops.prox_dual(x[s], u[s], y0[s], mask[s], mu)
        assert torch.equal(zz[s], z1) and torch.equal(uu[s], u1) and torch.equal(vv[s], v1)


def test_fft2c_rejects_sizes_outside_2_1024():
    from dt4image_restoration_b200._lib import PnpError
    for (h, w) in ((1025, 16), (16, 2048), (1, 64)):
        with pytest.raises(PnpError):
            ops.fft2c(torch.zeros(1, 1, h, w, dtype=torch.complex64, device=DEV))


# ------------------------------------------------------------------------------------------------
# prox + dual (env.py:87-93)
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B,H,W,kind,par,per_image_mu", [
    (2, 130, 130, "radial", 0.3, False), (3, 136, 120, "cartesian", 4, True), (2, 33, 47, "radial", 0.4, True),
    (1, 45, 51, "radial", 0.3, False), (2, 16, 24, "cartesian", 2, True), (1, 1024, 1024, "radial", 0.2, False)])
def test_prox_dual_any_size_matches_oracle(B, H, W, kind, par, per_image_mu):
    """The dense-DFT prox path (fftprox_any.cuh): same cases as the radix kernels at sizes the reference's step accepts."""
    batch = synth.make_batch(B, H, W, kind, par, sigma_n=5.0, seed0=H)
    st = O.reset(batch)
    g = torch.Generator().manual_seed(B + H)
    x = torch.rand(B, 1, H, W, generator=g)
    u = torch.complex(torch.randn(B, 1, H, W, generator=g), torch.randn(B, 1, H, W, generator=g)) * 0.1
    mu = (torch.rand(B, generator=g) * 0.9 + 0.05) if per_image_mu else torch.tensor([0.37])
    z_ref, u_ref = O.prox_dual(x, u, st["y0"], st["mask"], mu)
    z, un, v = ops.prox_dual(x.to(DEV), u.to(DEV), st["y0"].to(DEV), st["mask"].to(DEV), mu.to(DEV))
    tol = 2e-5 * max(1.0, np.log2(H * W) / 14)
    assert (z.cpu() - z_ref).abs().max() < tol
    assert (un.cpu() - u_ref).abs().max() < tol
    assert (v.cpu() - (z_ref - u_ref).real).abs().max() < 2 * tol
    # shared mask, u_out aliasing u_in (include/pnp_b200.h)
    ud = u.to(DEV).clone()
    zo, vo = torch.empty_like(ud), torch.empty(B, 1, H, W, device=DEV)
    ops.prox_dual(x.to(DEV), ud, st["y0"].to(DEV), st["mask"][:1].to(DEV), mu.to(DEV), out=(zo, ud, vo))
    z2_ref, u2_ref = O.prox_dual(x, u, st["y0"], st["mask"][:1], mu)
    assert (zo.cpu() - z2_ref).abs().max() < tol and (ud.cpu() - u2_ref).abs().max() < tol


@pytest.mark.parametrize("B,H,W,kind,par,per_image_mu", [
    (1, 128, 128, "radial", 0.3, False), (3, 256, 256, "cartesian", 4, True), (2, 64, 64, "radial", 0.2, True),
    (2, 512, 512, "cartesian", 8, False), (4, 32, 32, "cartesian", 4, True), (2, 64, 128, "radial", 0.3, False)])
def test_prox_dual_matches_oracle(B, H, W, kind, par, per_image_mu):
    batch = synth.make_batch(B, H, W, kind, par, sigma_n=5.0, seed0=H)
    st = O.reset(batch)
    g = torch.Generator().manual_seed(B + H)
    x = torch.rand(B, 1, H, W, generator=g)
    u = torch.complex(torch.randn(B, 1, H, W, generator=g), torch.randn(B, 1, H, W, generator=g)) * 0.1
    mu = (torch.rand(B, generator=g) * 0.9 + 0.05) if per_image_mu else torch.tensor([0.37])
    z_ref, u_ref = O.prox_dual(x, u, st["y0"], st["mask"], mu)
    z, un, v = ops.prox_dual(x.to(DEV), u.to(DEV), st["y0"].to(DEV), st["mask"].to(DEV), mu.to(DEV))
    assert (z.cpu() - z_ref).abs().max() < 2e-5
    assert (un.cpu() - u_ref).abs().max() < 2e-5
    assert (v.cpu() - (z_ref - u_ref).real).abs().max() < 4e-5
    # shared mask [1,1,H,W] with B>1 (extension; the reference raises IndexError there)
    z2, _, _ = ops.prox_dual(x.to(DEV), u.to(DEV), st["y0"].to(DEV), st["mask"][:1].to(DEV), mu.to(DEV))
    z2_ref, _ = O.prox_dual(x, u, st["y0"], st["mask"][:1], mu)
    assert (z2.cpu() - z2_ref).abs().max() < 2e-5


def test_prox_dual_properties_full_size():
    """Size-independent properties at BASELINE size: data consistency and linearity (mu -> inf keeps z = x+u)."""
    B, H, W = 8, 256, 256
    batch = synth.make_batch(B, H, W, "cartesian", 4, 0.0, seed0=0)
    st = O.reset(batch)
    y0, mask = st["y0"].to(DEV), st["mask"].to(DEV)
    g = torch.Generator().manual_seed(1)
    x = torch.rand(B, 1, H, W, generator=g).to(DEV)
    u = torch.zeros(B, 1, H, W, dtype=torch.complex64, device=DEV)
    # mu = 0: sampled k-space bins of z equal y0 exactly, the others equal fft(x)
    z, un, _ = ops.prox_dual(x, u, y0, mask, torch.zeros(1, device=DEV))
    Z = ops.fft2c(z)
    X = ops.fft2c(torch.complex(x, torch.zeros_like(x)))
    assert (Z - torch.where(mask, y0, X)).abs().max() < 5e-5
    # u' = u + x - z
    assert (un - (u + x - z)).abs().max() < 1e-6
    # huge mu: z -> x + u
    z_inf, _, _ = ops.prox_dual(x, u, y0, mask, torch.full((1,), 1e8, device=DEV))
    assert (z_inf - x).abs().max() < 1e-4


@pytest.mark.parametrize("case,B,H,W", [("cartesian_per_image", 5, 256, 256), ("cartesian_shared", 5, 256, 256),
                                        ("radial", 5, 256, 256), ("mixed", 5, 256, 256), ("rows_only", 5, 256, 256),
                                        ("cartesian_per_image", 3, 128, 128), ("radial", 3, 128, 128),
                                        ("cartesian_shared", 2, 512, 512), ("mixed", 2, 512, 512),
                                        ("cartesian_per_image", 4, 64, 128), ("rows_only", 4, 128, 64),
                                        # H != 256 with W == 256: the row mask must stay in the plain-byte layout
                                        ("cartesian_per_image", 3, 128, 256), ("cartesian_shared", 2, 512, 256),
                                        ("radial", 2, 128, 256), ("cartesian_per_image", 2, 256, 128)])
@pytest.mark.parametrize("per_image_mu", [False, True])
def test_prox_prepared_paths_match_oracle(case, B, H, W, per_image_mu):
    """Prepared prox: column-only masks take a row-only kernel (fftprox_sep.cuh), everything else the general kernels
    (cluster kernel at 256x256, three-launch path otherwise); the choice is made on the device and every path must
    equal the oracle (reference env.py:87-93)."""
    kind, par = ("radial", 0.3) if case == "radial" else ("cartesian", 4)
    batch = synth.make_batch(B, H, W, kind, par, sigma_n=10.0, seed0=3)
    st = O.reset(batch)
    mask = st["mask"].clone()
    if case == "mixed":
        mask[B // 2, 0, H // 3, :] = ~mask[B // 2, 0, H // 3, :]   # one image loses the column structure
    if case == "rows_only":                                      # fully sampled ROWS: not the row-only kernel's case
        mask = O.reset(synth.make_batch(B, W, H, kind, par, seed0=3))["mask"].transpose(-1, -2).contiguous()
    y0 = torch.where(mask, st["y0"], torch.zeros_like(st["y0"])) + 0.01 * (~mask) * st["y0"].roll(1, -1)
    if case == "cartesian_shared":
        mask = mask[:1]
    g = torch.Generator().manual_seed(11)
    x = torch.rand(B, 1, H, W, generator=g)
    u = torch.complex(torch.randn(B, 1, H, W, generator=g), torch.randn(B, 1, H, W, generator=g)) * 0.1
    mu = (torch.rand(B, generator=g) * 0.9 + 0.05) if per_image_mu else torch.tensor([0.37])
    z_ref, u_ref = O.prox_dual(x, u, y0, mask, mu)
    prep = ops.ProxPrepared(y0.to(DEV), mask.to(DEV))
    assert prep.column_only == case.startswith("cartesian")
    # kind -1: both kernels are launched and the device flag decides; None: the host-side hint (known after column_only's
    # synchronisation) launches only the kernel whose case it is
    for kind in (-1, None):
        z, un, v = prep.prox_dual(x.to(DEV), u.to(DEV), mu.to(DEV), kind=kind)
        assert (z.cpu() - z_ref).abs().max() < 2e-5
        assert (un.cpu() - u_ref).abs().max() < 2e-5
        assert (v.cpu() - (z_ref - u_ref).real).abs().max() < 4e-5
    # the one-shot entry point (general kernels) agrees
    z2, _, _ = ops.prox_dual(x.to(DEV), u.to(DEV), y0.to(DEV), mask.to(DEV), mu.to(DEV))
    assert (z2 - z).abs().max() < 2e-5


# ------------------------------------------------------------------------------------------------
# tensor-core 3x3 conv (noise.py:75-89)
# ------------------------------------------------------------------------------------------------
def conv_ref(in0, in1, w, b):
    x = in0 if in1 is None else torch.cat([in0, in1], dim=-1)
    x = x.float().permute(0, 3, 1, 2)
    y = F.leaky_relu(F.conv2d(x, bf16r(w), b, padding=1), 0.2)
    return y.permute(0, 2, 3, 1)


CONV_CASES = [
    # B, H, W, C0, C1, Cout
    (1, 16, 16, 32, 0, 32), (2, 32, 32, 32, 0, 32), (1, 32, 48, 32, 0, 64), (2, 32, 32, 64, 0, 64),
    (1, 16, 16, 64, 0, 128), (2, 16, 32, 128, 0, 128), (1, 16, 16, 128, 0, 256), (1, 16, 16, 256, 0, 512),
    (1, 16, 16, 512, 0, 512), (1, 32, 32, 32, 64, 32), (1, 32, 32, 64, 128, 64), (1, 16, 16, 128, 256, 128),
    (1, 16, 16, 256, 512, 256), (3, 40, 24, 32, 0, 32), (1, 8, 8, 256, 0, 512), (2, 20, 36, 64, 0, 64),
    (1, 256, 256, 32, 0, 32),
    # 32 output channels with >= 64 input channels: kw-stacked kernel (unet_conv_kws.cuh), 16x12 tiles, ragged edges
    (2, 40, 52, 32, 64, 32), (3, 20, 36, 64, 0, 32), (2, 19, 27, 32, 64, 32), (1, 256, 256, 32, 64, 32), (1, 16, 12, 64, 32, 32),
]


@pytest.fixture
def splitk_mode():
    """Set the conv kernel choice (0: ordinary kernels only, 1: split-K cluster kernel for every eligible conv, -1: auto) for
    one test and restore the previous mode afterwards."""
    from dt4image_restoration_b200 import _lib
    lib = _lib.lib()
    old = []

    def set_mode(mode):
        old.append(lib.pnp_unet_set_splitk(mode))
    yield set_mode
    if old:
        lib.pnp_unet_set_splitk(old[0])


@pytest.mark.parametrize("splitk", [0, 1])
@pytest.mark.parametrize("B,H,W,C0,C1,Cout", CONV_CASES + [(1, 64, 64, 128, 256, 128), (3, 16, 16, 64, 0, 64), (2, 24, 40, 256, 0, 256),
                                                            (1, 16, 16, 512, 256, 256)])
def test_conv3x3_umma_matches_fp32_reference(B, H, W, C0, C1, Cout, splitk, splitk_mode):
    splitk_mode(splitk)
    g = torch.Generator().manual_seed(C0 * 13 + Cout + H)
    in0 = (torch.randn(B, H, W, C0, generator=g)).to(torch.bfloat16)
    in1 = (torch.randn(B, H, W, C1, generator=g)).to(torch.bfloat16) if C1 else None
    cin = C0 + C1
    w = torch.randn(Cout, cin, 3, 3, generator=g) * (2.0 / (9 * cin)) ** 0.5
    b = torch.randn(Cout, generator=g) * 0.1
    ref = conv_ref(in0, in1, w, b)
    got = ops.conv3x3_bf16(in0.to(DEV), w.to(DEV), b.to(DEV), in1.to(DEV) if C1 else None).float().cpu()
    err = (got - ref).abs()
    tol = 1e-2 * ref.abs() + 2e-3            # bf16 output rounding (2^-9) + accumulation order
    assert bool((err <= tol).all()), f"max err {err.max().item()} at {np.unravel_index(err.argmax(), err.shape)}"


# ------------------------------------------------------------------------------------------------
# whole denoiser, layer by layer (noise.py:119-133, 155-164)
# ------------------------------------------------------------------------------------------------
def sd_to_cuda_denoiser(params):
    return UNetDenoiser2D(state_dict=params).to(DEV)


@pytest.mark.parametrize("splitk", [-1, 0])
@pytest.mark.parametrize("B,H,W,kind", [(2, 64, 64, "kaiming"), (1, 128, 128, "default"), (1, 256, 256, "kaiming"),
                                         (2, 48, 80, "kaiming"), (1, 36, 52, "kaiming")])
def test_unet_layerwise_against_oracle(B, H, W, kind, splitk, splitk_mode):
    splitk_mode(splitk)        # -1: the deep levels of these small batches run on the split-K cluster kernel; 0: ordinary kernels
    params = O.init_unet_params(1, kind)
    den = sd_to_cuda_denoiser(params)
    g = torch.Generator().manual_seed(H + W)
    v = torch.rand(B, 1, H, W, generator=g)
    sigma = torch.rand(B, generator=g) * 0.2 + 0.02
    taps = {}
    pre_ref = O.denoise(params, v, sigma, clamp=False, taps=taps)
    out, pre = den(v.to(DEV), sigma.to(DEV), preclamp=True)
    plan = den.plan(B, H, W)
    # layers whose buffers are not recycled by later layers
    for name in ["inc.conv-2", "down1.pooled", "down1.conv-2", "down2.pooled", "down2.conv-2", "down3.pooled", "down3.conv-2",
                 "down4.pooled", "down4.conv-0", "down4.conv-1", "down4.conv-2", "up1.upsampled", "up2.upsampled",
                 "up3.upsampled", "up4.upsampled"]:
        got = plan.activation(name).float().cpu().permute(0, 3, 1, 2)
        ref = taps[name]
        rel = (got - ref).norm() / (ref.norm() + 1e-12)
        assert rel < 2e-2, f"{name}: relative L2 error {rel.item():.3e}"
    resid_ref = pre_ref - v
    resid = pre.cpu() - v
    rel = (resid - resid_ref).norm() / (resid_ref.norm() + 1e-12)
    assert rel < 3e-2, f"residual relative L2 error {rel.item():.3e}"
    assert (out.cpu() - torch.clamp(pre_ref, 0, 1)).abs().max() < (1e-3 if kind == "default" else 2e-2)
    assert out.min() >= 0 and out.max() <= 1


@pytest.mark.parametrize("splitk", [0, -1])
def test_unet_micro_batched_plan_equals_whole_batch(splitk, splitk_mode):
    """A plan whose batch exceeds the workspace budget runs in micro-batches on one bounded workspace (SURVEY 7.3-5: B = 4096
    at 256x256 needs it); with the same kernels (split-K off) the results equal the whole-batch plan bit for bit; with the
    automatic kernel choice the small micro-batches run their deep levels on the split-K kernel (another summation order)."""
    import ctypes as C
    splitk_mode(splitk)
    from dt4image_restoration_b200 import _lib
    l = _lib.lib()
    B, H, W = 11, 64, 64
    params = O.init_unet_params(2, "kaiming")
    g = torch.Generator().manual_seed(3)
    v = torch.rand(B, 1, H, W, generator=g).to(DEV)
    sg = (torch.rand(B, generator=g) * 0.2 + 0.02).to(DEV)
    den = UNetDenoiser2D(state_dict=params).to(DEV)
    whole = den.plan(B, H, W)
    assert l.pnp_unet_micro_batch(whole.handle) == B
    ref = whole.forward(v, sg).clone()
    old = l.pnp_unet_set_workspace_cap(l.pnp_unet_workspace_bytes(4, H, W))
    try:
        den2 = UNetDenoiser2D(state_dict=params).to(DEV)
        small = den2.plan(B, H, W)
        mb = l.pnp_unet_micro_batch(small.handle)
        assert 1 <= mb <= 4 and small.workspace.numel() <= l.pnp_unet_workspace_bytes(4, H, W)
        assert l.pnp_unet_num_launches(small.handle) > l.pnp_unet_num_launches(whole.handle)
        out = small.forward(v, sg)
        if splitk == 0:
            assert torch.equal(out, ref)
        else:
            assert (out - ref).abs().max() < 5e-3
    finally:
        l.pnp_unet_set_workspace_cap(old)


def test_unet_golden_odd_sizes(golden_dir):
    """Reference outputs (fixtures) for the `up` pad path (noise.py:49-53)."""
    gd = np.load(os.path.join(golden_dir, "ref_unet_kaiming.npz"))
    params = O.init_unet_params(1, "kaiming")
    den = sd_to_cuda_denoiser(params)
    gen = torch.Generator().manual_seed(99)
    for (h, w) in ((64, 64), (48, 80), (36, 52)):
        inp = torch.rand(2, 2, h, w, generator=gen)
        # the golden net input has an arbitrary second channel; ours synthesises a constant sigma map, so
        # compare on a constant-map input instead and use the oracle (pinned to the same fixture) as bridge
        ref_fixture = torch.from_numpy(gd[f"out_{h}x{w}"])
        assert (O.unet_forward(params, inp) - ref_fixture).abs().max() < 1e-5
        sig = torch.tensor([0.07, 0.15])
        inp_c = torch.cat([inp[:, :1], torch.ones(2, 1, h, w) * sig.view(2, 1, 1, 1)], dim=1)
        ref = O.unet_forward(params, inp_c)
        _, pre = den(inp[:, :1].to(DEV), sig.to(DEV), preclamp=True)
        r_ref, r_got = ref - inp[:, :1], pre.cpu() - inp[:, :1]
        assert (r_got - r_ref).norm() / r_ref.norm() < 3e-2


@pytest.mark.parametrize("pair", ["0", "1"])
def test_conv3x3_cta_pair_variant_matches_reference(pair):
    """The CTA-pair kernel (unet_conv_pair.cuh, tcgen05.mma.cta_group::2) is used by default for layers with streamed
    weights; PNP_CONV_PAIR=1 forces it for every eligible layer, =0 forces the single-CTA kernel.  Both must compute the
    same convolutions; the switch is read once per process, hence the subprocess."""
    import os, subprocess, sys
    code = r'''
import torch, numpy as np, torch.nn.functional as F
from dt4image_restoration_b200 import ops
bf16r = lambda t: t.to(torch.bfloat16).float()
for (B, H, W, C0, C1, Cout) in [(2, 32, 32, 64, 0, 64), (1, 16, 16, 64, 0, 128), (3, 40, 24, 64, 128, 64), (1, 16, 16, 256, 512, 256),
                                (2, 20, 36, 32, 0, 64), (5, 16, 16, 128, 0, 128)]:
    g = torch.Generator().manual_seed(C0 + Cout + H)
    in0 = torch.randn(B, H, W, C0, generator=g).to(torch.bfloat16)
    in1 = torch.randn(B, H, W, C1, generator=g).to(torch.bfloat16) if C1 else None
    cin = C0 + C1
    w = torch.randn(Cout, cin, 3, 3, generator=g) * (2.0 / (9 * cin)) ** 0.5
    b = torch.randn(Cout, generator=g) * 0.1
    x = in0 if in1 is None else torch.cat([in0, in1], dim=-1)
    ref = F.leaky_relu(F.conv2d(x.float().permute(0, 3, 1, 2), bf16r(w), b, padding=1), 0.2).permute(0, 2, 3, 1)
    got = ops.conv3x3_bf16(in0.cuda(), w.cuda(), b.cuda(), in1.cuda() if C1 else None).float().cpu()
    err = (got - ref).abs()
    assert bool((err <= 1e-2 * ref.abs() + 2e-3).all()), (B, H, W, C0, C1, Cout, err.max().item())
print("pair ok")
'''
    env = dict(os.environ, PNP_CONV_PAIR=pair)
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-c", code], cwd=root, env=env, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "pair ok" in r.stdout, r.stdout + r.stderr


def test_psnr_allgather_single_rank_protocol():
    """Fused reward + peer all-gather kernel with a world of one: values equal pnp_psnr bit for bit, the arrival counter and
    the double buffering advance per call, ragged batches are accepted, no timeout."""
    from dt4image_restoration_b200.dist import PeerRewardGather
    pg = PeerRewardGather(7, "cuda", local_only=True)
    prev = None
    for it, B in enumerate([7, 5, 7, 1]):
        g = torch.Generator(device="cuda").manual_seed(it)
        x = torch.rand(B, 1, 64, 64, device="cuda", generator=g) * 1.2 - 0.1
        gt = torch.rand(B, 1, 64, 64, device="cuda", generator=g)
        allr = pg.psnr_allgather(x, gt)
        assert allr.shape == (1, 7)
        assert torch.equal(allr[0, :B], ops.psnr(x, gt).reshape(-1).to(allr.device))
        if prev is not None:                      # the previous call's results are still intact (other parity)
            assert torch.equal(prev[0], prev[1])
        prev = (allr[0, :B], allr[0, :B].clone())
    assert not pg.timed_out()
    assert int(pg.buf.view(torch.int32)[pg.flag_word].item()) == 4 and int(pg.local[0].item()) == 20


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_psnr_allgather_two_ranks_matches_nccl():
    import os, subprocess, sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
                        "127.0.0.1", "--master-port", "29611", os.path.join(root, "tools", "peer_gather_check.py")],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert "match_nccl=True" in r.stdout


@pytest.mark.parametrize("B,S,kind", [(45, 256, "radial"), (31, 256, "random"), (160, 128, "radial"), (150, 128, "cartesian")])
def test_prox_cluster_kernels_multi_round_batches(B, S, kind):
    """Batches larger than the number of resident clusters (14 at 256x256, 71-74 at 128x128): every cluster processes
    several images back to back, which exercises the bulk-load prefetch of the NEXT image, the mbarrier phase flips and the
    reuse of the exchange buffers across images.  Per-image masks and per-image mu, every image checked against the oracle."""
    g = torch.Generator().manual_seed(B + S)
    x = torch.rand(B, 1, S, S, generator=g)
    u = torch.complex(torch.randn(B, 1, S, S, generator=g), torch.randn(B, 1, S, S, generator=g)) * 0.1
    y0 = torch.complex(torch.randn(B, 1, S, S, generator=g), torch.randn(B, 1, S, S, generator=g))
    if kind == "radial":
        base = torch.from_numpy(synth.radial_mask(S, S, 0.3)).bool()
        mask = torch.stack([torch.roll(base, shifts=(b % 5, (3 * b) % 7), dims=(0, 1)) for b in range(B)]).reshape(B, 1, S, S)
    elif kind == "random":
        mask = torch.rand(B, 1, S, S, generator=g) < 0.25
    else:
        mask = (torch.rand(B, 1, 1, S, generator=g) < 0.3).expand(B, 1, S, S).contiguous()
    mu = torch.rand(B, generator=g) * 0.9 + 0.05
    z_ref, u_ref = O.prox_dual(x, u, y0, mask, mu)
    prep = ops.ProxPrepared(y0.to(DEV), mask.to(DEV))
    for it in range(2):
        z, un, v = prep.prox_dual(x.to(DEV), u.to(DEV), mu.to(DEV))
        assert (z.cpu() - z_ref).abs().amax(dim=(1, 2, 3)).max() < 2e-5, f"call {it}"
        assert (un.cpu() - u_ref).abs().max() < 2e-5
        assert (v.cpu() - (z_ref - u_ref).real).abs().max() < 4e-5
    # u_out aliasing u_in (the engine's calling convention)
    u_io = u.to(DEV).clone()
    z2, _, _ = prep.prox_dual(x.to(DEV), u_io, mu.to(DEV), out=(torch.empty_like(u_io), u_io, torch.empty(B, 1, S, S, device=DEV)))
    assert (z2.cpu() - z_ref).abs().max() < 2e-5 and (u_io.cpu() - u_ref).abs().max() < 2e-5
