"""pnp_ssim (csrc/ssim.cu) through ops.ssim, PnPEngine.ssim and PnPEnv.compute_ssim against the float64 reference
(tests/ssim_reference.py): |diff| <= 1e-5 per image, bitwise determinism, batch independence, graph capture, rejection."""
import numpy as np
import pytest
import torch

from dt4image_restoration_b200 import _lib, ops, synth
from dt4image_restoration_b200.engine import PnPEngine
from dt4image_restoration_b200.env import PnPEnv
from dt4image_restoration_b200.noise import UNetDenoiser2D
from oracle import pnp_oracle as O
from ssim_reference import ssim as ssim_ref

pytestmark = pytest.mark.gpu
DEV = "cuda"
TOL = 1e-5

SHAPES = [(1, 11, 11), (3, 16, 16), (2, 45, 51), (4, 130, 130), (2, 136, 120), (64, 128, 128), (64, 256, 256),
          (4, 512, 512), (1, 1024, 1024), (1, 2000, 37)]


def _random(B, H, W, seed):
    g = torch.Generator().manual_seed(seed)
    x = torch.rand(B, 1, H, W, generator=g) * 1.4 - 0.2
    gt = torch.rand(B, 1, H, W, generator=g)
    return x, gt


def _phantom(B, H, W, seed):
    rng = np.random.default_rng(seed)
    gt = np.stack([synth.phantom(H, W, seed + b) for b in range(B)])[:, None]
    x = gt + rng.normal(0.0, 0.05, gt.shape)
    return torch.from_numpy(x.astype(np.float32)), torch.from_numpy(gt.astype(np.float32))


def _checkerboard(B, H, W, seed):
    i, j = np.meshgrid(np.arange(H), np.arange(W), indexing="ij")
    cb = ((i + j) % 2).astype(np.float32)
    rng = np.random.default_rng(seed)
    x = np.broadcast_to(cb, (B, 1, H, W)).copy()
    gt = np.clip(x * 0.9 + 0.05 + rng.normal(0.0, 0.02, x.shape), 0, 1)
    return torch.from_numpy(x), torch.from_numpy(gt.astype(np.float32))


def _constant(B, H, W, seed):
    x = torch.full((B, 1, H, W), 0.3) + 0.1 * torch.arange(B).reshape(B, 1, 1, 1)
    return x, torch.full((B, 1, H, W), 0.7)


def _check(x, gt):
    got = ops.ssim(x.to(DEV), gt.to(DEV))
    assert got.shape == (x.shape[0],) and got.dtype == torch.float32 and got.is_cuda
    ref = ssim_ref(x, gt)[:, 0]
    err = (got.cpu().double() - ref).abs().max().item()
    assert err <= TOL, err
    return got


@pytest.mark.parametrize("B,H,W", SHAPES)
def test_random_against_reference(B, H, W):
    _check(*_random(B, H, W, seed=B * 7 + H * 3 + W))


@pytest.mark.parametrize("make", [_phantom, _checkerboard, _constant])
@pytest.mark.parametrize("B,H,W", [(2, 45, 51), (4, 256, 256)])
def test_structured_inputs_against_reference(make, B, H, W):
    _check(*make(B, H, W, seed=H + W))


def test_constant_pair_gives_one():
    x = torch.full((2, 1, 64, 64), 0.42)
    assert (ops.ssim(x.to(DEV), x.to(DEV)) - 1).abs().max().item() <= 1e-6


def test_shared_gt():
    x, gt = _random(5, 130, 136, seed=1)
    got = _check(x, gt[0, 0])
    per_image = ops.ssim(x.to(DEV), gt[0:1].expand(5, -1, -1, -1).contiguous().to(DEV))
    assert torch.equal(got, per_image)


def test_unaligned_base_pointer():
    x, gt = _random(5, 45, 51, seed=2)                 # H*W = 2295 floats: image 1 starts 4 bytes past a 16-byte boundary
    xd, gd = x.to(DEV)[1:], gt.to(DEV)[1:]
    assert xd.data_ptr() % 16 != 0 and gd.data_ptr() % 16 != 0
    got = ops.ssim(xd, gd)
    assert (got.cpu().double() - ssim_ref(x[1:], gt[1:])[:, 0]).abs().max().item() <= TOL
    xc, gc = _random(5, 256, 256, seed=3)
    xs, gs = xc.to(DEV).reshape(-1)[3:3 + 4 * 65536], gc.to(DEV).reshape(-1)[1:1 + 4 * 65536]
    got = ops.ssim(xs.reshape(4, 256, 256), gs.reshape(4, 256, 256))
    ref = ssim_ref(xc.reshape(-1)[3:3 + 4 * 65536].reshape(4, 256, 256), gc.reshape(-1)[1:1 + 4 * 65536].reshape(4, 256, 256))
    assert (got.cpu().double() - ref[:, 0]).abs().max().item() <= TOL


def test_same_address_gives_one():
    x = torch.rand(3, 1, 77, 93, generator=torch.Generator().manual_seed(4)).to(DEV)
    assert (ops.ssim(x, x) - 1).abs().max().item() <= 1e-6


def test_deterministic_and_batch_independent():
    x, gt = _random(64, 256, 256, seed=5)
    xd, gd = x.to(DEV), gt.to(DEV)
    a, b = ops.ssim(xd, gd), ops.ssim(xd, gd)
    assert torch.equal(a, b)
    for i in (0, 17, 63):
        assert torch.equal(ops.ssim(xd[i:i + 1], gd[i:i + 1]), a[i:i + 1])
    shared = ops.ssim(xd, gd[0])
    assert torch.equal(ops.ssim(xd[40:41], gd[0]), shared[40:41])


@pytest.fixture(scope="module")
def engine():
    B, H, W = 3, 64, 64
    eng = PnPEngine(UNetDenoiser2D(state_dict=O.init_unet_params(1, "kaiming")), B, H, W, DEV)
    batch = synth.make_batch(B, H, W, "radial", 0.3, 5.0, seed0=7)
    eng.reset({k: torch.from_numpy(np.ascontiguousarray(v)) for k, v in batch.items()})
    eng.set_actions(0.1, 0.5)
    for _ in range(3):
        eng.step()
    torch.cuda.synchronize()
    return eng


def test_engine_ssim_matches_ops_and_env(engine):
    got = engine.ssim()
    assert got.data_ptr() == engine.ssim_out.data_ptr()
    assert torch.equal(got, ops.ssim(engine.x, engine.gt))
    assert (got.cpu().double() - ssim_ref(engine.x.cpu(), engine.gt.cpu())[:, 0]).abs().max().item() <= TOL
    env_vals = PnPEnv.compute_ssim(engine.x, engine.gt)
    assert env_vals.shape == (3, 1) and env_vals.device.type == "cpu"
    assert torch.equal(env_vals[:, 0], got.cpu())
    assert torch.equal(PnPEnv.compute_ssim(engine.x.cpu(), engine.gt.cpu()), env_vals)


def test_engine_ssim_graph_capture(engine):
    eager = engine.ssim().clone()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        engine.ssim()
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = engine.ssim()
    engine.ssim_out.zero_()
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(out, eager)


def test_rejection():
    lib = _lib.lib()
    x = torch.rand(2, 16, 16, device=DEV)
    out = torch.empty(2, device=DEV)
    work = ops.aligned_empty(4096, DEV, align=16)
    args = lambda B, H, W: (x.data_ptr(), x.data_ptr(), H * W, out.data_ptr(), work.data_ptr(), B, H, W, _lib.stream_ptr())
    assert lib.pnp_ssim(*args(2, 16, 16)) == 0
    assert lib.pnp_ssim(*args(2, 10, 16)) < 0
    assert lib.pnp_ssim(*args(2, 16, 10)) < 0
    assert lib.pnp_ssim(*args(0, 16, 16)) < 0
    assert lib.pnp_ssim(None, x.data_ptr(), 256, out.data_ptr(), work.data_ptr(), 2, 16, 16, _lib.stream_ptr()) < 0
    assert lib.pnp_ssim(x.data_ptr(), x.data_ptr(), 256, out.data_ptr(), None, 2, 16, 16, _lib.stream_ptr()) < 0
    assert b"pnp_ssim" in lib.pnp_last_error()
    with pytest.raises(_lib.PnpError):
        ops.ssim(torch.rand(2, 16, 16), torch.rand(2, 16, 16))
    with pytest.raises(_lib.PnpError):
        ops.ssim(torch.rand(1, 10, 10, device=DEV), torch.rand(1, 10, 10, device=DEV))
