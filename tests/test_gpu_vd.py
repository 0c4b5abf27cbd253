"""pnp_variable_density_masks (csrc/measure.cuh) through ops, ops.make_items and PnPEngine.reset_from_gt against the float64
reference (tests/vd_reference.py): masks bit for bit at 14 shapes, four powers, per-image and scalar accelerations, extreme
seeds, the straddling-tie seeds and the ACS extremes; batch-position independence, determinism, graph capture, batches over
65535, unaligned outputs, the engine entry point with the prox routing of these masks, rejection."""
import numpy as np
import pytest
import torch

from dt4image_restoration_b200 import _lib, ops, synth
from dt4image_restoration_b200.engine import PnPEngine
from dt4image_restoration_b200.noise import UNetDenoiser2D
from oracle import pnp_oracle as O
from vd_reference import acs_size, vd_mask

pytestmark = pytest.mark.gpu
DEV = "cuda"
SHAPES = [(2, 3), (3, 2), (16, 16), (30, 34), (45, 51), (64, 48), (128, 128), (130, 130), (136, 120), (256, 256),
          (512, 512), (1000, 1000), (1024, 1024), (1024, 37)]
SEEDS = [0, 1, 7, (1 << 40) + 3, -5, (1 << 63) - 1]      # -5: an int64 seed is used as its uint64 bit pattern
ACCELS = [4, 2, 8, 3, 1, 0]                               # 1 and 0: every pixel
TIE_SEEDS = [533, 1284]                                   # 256^2, accel 2, power 0, 20x20 ACS (tests/test_vd_reference.py)


def _vd(B, H, W, accel, seeds, power=3, acs_frac=0.08, out=None):
    return ops.variable_density_masks(B, H, W, accel, seeds, power=power, acs_frac=acs_frac, out=out).cpu().numpy()


def _ref(H, W, accel, seed, power=3, acs=None):
    ah, aw = acs if acs is not None else (acs_size(H), acs_size(W))
    return vd_mask(H, W, accel, seed, power, ah, aw)


@pytest.mark.parametrize("H,W", SHAPES)
@pytest.mark.parametrize("power", [0, 1, 3, 8])
def test_masks_equal_reference(H, W, power):
    acc = torch.tensor(ACCELS, dtype=torch.int32, device=DEV)
    got = _vd(6, H, W, acc, torch.tensor(SEEDS, dtype=torch.int64, device=DEV), power)
    assert got.dtype == np.uint8 and got.shape == (6, H, W)
    for b in range(6):
        assert np.array_equal(got[b], _ref(H, W, ACCELS[b], SEEDS[b], power)), b
    s0 = _vd(3, H, W, 4, 40, power)                       # scalar accel, int s0 = s0 + arange(B)
    for b in range(3):
        assert np.array_equal(s0[b], _ref(H, W, 4, 40 + b, power)), b


@pytest.mark.parametrize("seed", TIE_SEEDS)
def test_straddling_tie_seeds(seed):
    got = _vd(1, 256, 256, 2, torch.tensor([seed], dtype=torch.int64, device=DEV), power=0)
    assert np.array_equal(got[0], _ref(256, 256, 2, seed, 0))


@pytest.mark.parametrize("H,W", [(2, 3), (45, 51), (256, 256), (1024, 37), (1024, 1024)])
def test_acs_extremes(H, W):
    seeds = torch.tensor([3, 4], dtype=torch.int64, device=DEV)
    lib = _lib.lib()
    acc = torch.tensor([4, 2], dtype=torch.int32, device=DEV)
    for ah, aw in ((0, 0), (1, 1), (H, W), (H, W - W // 3), (1, W), (H, 1)):
        out = torch.empty(2, H, W, dtype=torch.uint8, device=DEV)
        _lib.check(lib.pnp_variable_density_masks(acc.data_ptr(), 1, seeds.data_ptr(), ah, aw, 3, out.data_ptr(), 2, H, W,
                                                  _lib.stream_ptr()))
        got = out.cpu().numpy()
        for b, a in enumerate((4, 2)):
            assert np.array_equal(got[b], vd_mask(H, W, a, 3 + b, 3, ah, aw)), (ah, aw, b)
    for frac in (0.0, 1.0, 0.5):                           # acs_frac 0 still gives a 1x1 block
        got = _vd(2, H, W, 4, 9, acs_frac=frac)
        ah, aw = max(1, int(round(frac * H))), max(1, int(round(frac * W)))
        for b in range(2):
            assert np.array_equal(got[b], _ref(H, W, 4, 9 + b, 3, (ah, aw))), (frac, b)


@pytest.mark.parametrize("H,W", [(256, 256), (45, 51), (1024, 1024), (512, 512)])
def test_batch_position_independence_and_determinism(H, W):
    B = 5
    acc = torch.tensor([4, 2, 8, 4, 3], dtype=torch.int32, device=DEV)
    seeds = torch.tensor([3, -8, 11, 12, (1 << 50)], dtype=torch.int64, device=DEV)
    m = _vd(B, H, W, acc, seeds)
    assert np.array_equal(m, _vd(B, H, W, acc, seeds))
    for b in range(B):
        assert np.array_equal(_vd(1, H, W, acc[b:b + 1], seeds[b:b + 1])[0], m[b]), b
    perm = torch.tensor([4, 2, 0, 3, 1], device=DEV)
    assert np.array_equal(_vd(B, H, W, acc[perm], seeds[perm]), m[perm.cpu().numpy()])
    big = _vd(300, H, W, acc.repeat(60), seeds.repeat(60))      # another cluster size than B = 1 and B = 5
    assert np.array_equal(big[295:], m) and np.array_equal(big[:5], m)


@pytest.mark.parametrize("H,W,offset", [(45, 51, 1), (256, 256, 3), (2, 3, 7), (1024, 37, 9)])
def test_unaligned_output(H, W, offset):
    B = 3
    buf = torch.full((B * H * W + offset + 16,), 7, dtype=torch.uint8, device=DEV)
    out = buf[offset:offset + B * H * W].view(B, H, W)
    got = _vd(B, H, W, 4, 5, out=out)
    for b in range(B):
        assert np.array_equal(got[b], _ref(H, W, 4, 5 + b))
    rest = buf.cpu().numpy()
    assert np.all(rest[:offset] == 7) and np.all(rest[offset + B * H * W:] == 7)


@pytest.mark.parametrize("H,W", [(256, 256), (130, 130)])
def test_graph_capture(H, W):
    B = 3
    acc = torch.tensor([4, 2, 8], dtype=torch.int32, device=DEV)
    seeds = torch.tensor([5, 6, 7], dtype=torch.int64, device=DEV)
    mask = torch.empty(B, H, W, dtype=torch.uint8, device=DEV)

    def body():
        ops.variable_density_masks(B, H, W, acc, seeds, out=mask)

    body()
    eager = mask.clone()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        body()
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        body()
    mask.zero_()
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(eager, mask)


def test_batch_over_65535():
    B, H, W = 65537, 16, 16
    seeds = torch.arange(B, dtype=torch.int64, device=DEV) * 3 - 7
    acc = (torch.arange(B, device=DEV) % 7 + 1).to(torch.int32)
    m = _vd(B, H, W, acc, seeds)
    for b in (0, 1, 65535, B - 1):
        assert np.array_equal(m[b], _ref(H, W, int(acc[b]), int(seeds[b]))), b
    assert np.array_equal(m.reshape(B, -1).sum(1), np.maximum((H * W) // acc.cpu().numpy(), 1))


def test_make_items_vd_layout():
    H, W = 64, 48
    items = ops.make_items(torch.rand(H, W, device=DEV), torch.tensor([0.0, 5.0], device=DEV), 3, vd=4)
    ref = synth.make_batch(2, H, W, "cartesian", 4, 5.0, seed0=3)
    for k, v in ref.items():
        assert items[k].shape == v.shape and items[k].dtype == torch.from_numpy(v).dtype and items[k].is_cuda, k
    for b in range(2):
        assert np.array_equal(items["mask"][b].cpu().numpy(), _ref(H, W, 4, 3 + b))


@pytest.mark.parametrize("H,W", [(256, 256), (130, 130)])
def test_engine_reset_from_gt_equals_reset_of_make_items(H, W):
    B = 3
    params = O.init_unet_params(0, "default")
    den = UNetDenoiser2D(state_dict=params)
    gt = torch.rand(B, 1, H, W, device=DEV)
    a, b = PnPEngine(den, B, H, W, DEV), PnPEngine(den, B, H, W, DEV)
    a.reset_from_gt(gt, 10.0, 17, vd=4)
    b.reset(ops.make_items(gt, 10.0, 17, vd=4))
    names = ["x", "v", "z", "u", "y0", "mask", "gt"] + (["y0T", "maskT"] if a.prepared else [])
    for n in names:
        assert torch.equal(getattr(a, n), getattr(b, n)), n
    for k in range(B):
        assert np.array_equal(a.mask[k, 0].cpu().numpy(), _ref(H, W, 4, 17 + k))
    if (H, W) == (256, 256):
        assert a.prepared
        torch.cuda.synchronize()
        assert a.probe.get() == 0 and b.probe.get() == 0          # general masks: the cluster prox kernel
    for e in (a, b):
        e.set_actions(torch.tensor([0.1, 0.15, 0.2]), 0.5)
    for _ in range(3):
        a.step()
        b.step()
    for n in ("x", "z", "u", "v"):
        assert torch.equal(getattr(a, n), getattr(b, n)), n
    if (H, W) == (256, 256):
        a.reset_from_gt(gt, 10.0, 17, vd=1)                         # every pixel sampled: column-only, the row kernel
        torch.cuda.synchronize()
        assert bool(a.mask.all()) and a.probe.get() == 1
    with pytest.raises(ValueError):
        a.reset_from_gt(gt, 10.0, 17, accel=4, vd=4)


def test_rejection():
    H = W = 32
    acc = torch.full((2,), 4, dtype=torch.int32, device=DEV)
    seeds = torch.zeros(2, dtype=torch.int64, device=DEV)
    with pytest.raises(_lib.PnpError):
        ops.variable_density_masks(2, H, W, acc.cpu(), seeds)
    with pytest.raises(_lib.PnpError):
        ops.variable_density_masks(2, H, W, acc, seeds.cpu())
    with pytest.raises(_lib.PnpError):
        ops.variable_density_masks(2, H, W, acc, seeds, out=torch.empty(2, H, W, dtype=torch.uint8))
    with pytest.raises(_lib.PnpError):
        ops.variable_density_masks(2, 1030, W, 4, 0)
    with pytest.raises(_lib.PnpError):
        ops.variable_density_masks(2, H, W, 4, 0, power=17)
    with pytest.raises(TypeError):
        ops.variable_density_masks(2, H, W, acc.float(), seeds)
    with pytest.raises(ValueError):
        ops.make_items(torch.rand(2, H, W, device=DEV), 0.0, 0, accel=4, vd=4)
    lib = _lib.lib()
    out = torch.empty(2, H, W, dtype=torch.uint8, device=DEV)
    st = _lib.stream_ptr()
    assert lib.pnp_variable_density_masks(acc.data_ptr(), 1, seeds.data_ptr(), 3, 3, 3, out.data_ptr(), 2, H, W, st) == 0
    for args in ((acc.data_ptr(), 1, seeds.data_ptr(), 3, 3, 3, acc.data_ptr(), 2, H, W, st),
                 (acc.data_ptr(), 1, seeds.data_ptr(), 3, 3, 3, out.data_ptr(), 0, H, W, st),
                 (acc.data_ptr(), 1, seeds.data_ptr(), 33, 3, 3, out.data_ptr(), 2, H, W, st)):
        assert lib.pnp_variable_density_masks(*args) < 0
        assert b"pnp_variable_density_masks" in lib.pnp_last_error()
    torch.cuda.synchronize()
