"""pnp_radial_masks (csrc/measure.cuh) through ops, ops.make_items and PnPEngine.reset_from_gt against synth.radial_mask and
the float64 reference (tests/radial_reference.py): masks and line counts bit for bit, seeds and per-image fractions,
batch-position independence, determinism, graph capture, batches over 65535, unaligned outputs, the engine entry point and
the prox routing of radial masks, rejection."""
import numpy as np
import pytest
import torch

from dt4image_restoration_b200 import _lib, ops, synth
from dt4image_restoration_b200.engine import PnPEngine
from dt4image_restoration_b200.noise import UNetDenoiser2D
from oracle import pnp_oracle as O
from radial_reference import radial_mask

pytestmark = pytest.mark.gpu
DEV = "cuda"
SHAPES = [(2, 3), (3, 2), (16, 16), (30, 34), (45, 51), (64, 48), (128, 128), (130, 130), (136, 120), (256, 256),
          (512, 512), (1000, 1000), (1024, 1024), (1024, 37)]
FRACS = [0.05, 0.2, 0.3, 0.5, 1.0]
SEEDS = [0, 1, 7, (1 << 40) + 3, -5, (1 << 63) - 1]      # -5: an int64 seed is used as its uint64 bit pattern


def _radial(B, H, W, frac, seeds=None, out=None):
    lines = torch.full((B,), -1, dtype=torch.int32, device=DEV)
    m = ops.radial_masks(B, H, W, frac, seeds, out=out, lines_out=lines)
    return m.cpu().numpy(), lines.cpu().numpy()


@pytest.mark.parametrize("H,W", SHAPES)
def test_unseeded_masks_equal_synth_radial_mask(H, W):
    frac = torch.tensor(FRACS, dtype=torch.float64, device=DEV)
    got, lines = _radial(len(FRACS), H, W, frac)
    assert got.dtype == np.uint8 and got.shape == (len(FRACS), H, W)
    for b, f in enumerate(FRACS):
        ref, n = radial_mask(H, W, f)
        assert np.array_equal(got[b], ref) and lines[b] == n, f
        if H * W <= 512 * 512:                           # the CPU suite pins the reference to synth at every shape
            assert np.array_equal(got[b], synth.radial_mask(H, W, f)), f
    shared, _ = _radial(2, H, W, 0.3)                    # one frac for the batch (stride 0)
    assert np.array_equal(shared[0], got[2]) and np.array_equal(shared[1], got[2])


@pytest.mark.parametrize("H,W", [(2, 3), (45, 51), (130, 130), (256, 256), (1024, 37), (1024, 1024)])
def test_seeded_masks_equal_reference(H, W):
    fr = [0.3, 0.2, 0.05, 0.5, 1.0, 0.3]
    got, lines = _radial(6, H, W, torch.tensor(fr, dtype=torch.float64, device=DEV),
                         torch.tensor(SEEDS, dtype=torch.int64, device=DEV))
    for b in range(6):
        ref, n = radial_mask(H, W, fr[b], SEEDS[b])
        assert np.array_equal(got[b], ref) and lines[b] == n, b
    s0, _ = _radial(3, H, W, 0.3, 40)                    # int s0 = s0 + arange(B)
    for b in range(3):
        assert np.array_equal(s0[b], radial_mask(H, W, 0.3, 40 + b)[0])


def test_special_fractions():
    H, W = 64, 48
    fr = [0.0, -1.0, float("nan"), 1.5, float("inf"), 1e-12]
    got, lines = _radial(6, H, W, torch.tensor(fr, dtype=torch.float64, device=DEV), 9)
    for b in range(6):
        ref, n = radial_mask(H, W, fr[b], 9 + b)
        assert np.array_equal(got[b], ref) and lines[b] == n, fr[b]
    assert list(lines[:3]) == [0, 0, 0] and not got[:3].any()
    assert lines[3] == lines[4] == 8 * 64 and lines[5] == 1


@pytest.mark.parametrize("H,W", [(256, 256), (45, 51), (1024, 1024)])
def test_batch_position_independence_and_determinism(H, W):
    B = 5
    fr = torch.tensor([0.2, 0.3, 0.05, 0.5, 0.3], dtype=torch.float64, device=DEV)
    seeds = torch.tensor([3, -8, 11, 12, (1 << 50)], dtype=torch.int64, device=DEV)
    m, lines = _radial(B, H, W, fr, seeds)
    m2, lines2 = _radial(B, H, W, fr, seeds)
    assert np.array_equal(m, m2) and np.array_equal(lines, lines2)
    for b in range(B):
        one, n1 = _radial(1, H, W, fr[b:b + 1], seeds[b:b + 1])
        assert np.array_equal(one[0], m[b]) and n1[0] == lines[b], b
    perm = torch.tensor([4, 2, 0, 3, 1], device=DEV)
    mp, lp = _radial(B, H, W, fr[perm], seeds[perm])
    assert np.array_equal(mp, m[perm.cpu().numpy()]) and np.array_equal(lp, lines[perm.cpu().numpy()])


@pytest.mark.parametrize("H,W,offset", [(45, 51, 1), (256, 256, 3), (2, 3, 7), (1024, 37, 9)])
def test_unaligned_output(H, W, offset):
    B = 3
    buf = torch.full((B * H * W + offset + 16,), 7, dtype=torch.uint8, device=DEV)
    out = buf[offset:offset + B * H * W].view(B, H, W)
    got, _ = _radial(B, H, W, 0.3, 5, out=out)
    for b in range(B):
        assert np.array_equal(got[b], radial_mask(H, W, 0.3, 5 + b)[0])
    rest = buf.cpu().numpy()
    assert np.all(rest[:offset] == 7) and np.all(rest[offset + B * H * W:] == 7)


@pytest.mark.parametrize("H,W", [(256, 256), (130, 130)])
def test_graph_capture(H, W):
    B = 3
    fr = torch.tensor([0.2, 0.3, 0.5], dtype=torch.float64, device=DEV)
    seeds = torch.tensor([5, 6, 7], dtype=torch.int64, device=DEV)
    mask = torch.empty(B, H, W, dtype=torch.uint8, device=DEV)
    lines = torch.empty(B, dtype=torch.int32, device=DEV)

    def body():
        ops.radial_masks(B, H, W, fr, seeds, out=mask, lines_out=lines)

    body()
    eager = (mask.clone(), lines.clone())
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        body()
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        body()
    mask.zero_()
    lines.zero_()
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(eager[0], mask) and torch.equal(eager[1], lines)


def test_batch_over_65535():
    B, H, W = 65537, 16, 16
    seeds = torch.arange(B, dtype=torch.int64, device=DEV) * 3 - 7
    fr = (torch.arange(B, dtype=torch.float64, device=DEV) % 7 + 1) / 8
    m, lines = _radial(B, H, W, fr, seeds)
    for b in (0, 1, 65535, B - 1):
        ref, n = radial_mask(H, W, float(fr[b]), int(seeds[b]))
        assert np.array_equal(m[b], ref) and lines[b] == n, b
        one, n1 = _radial(1, H, W, fr[b:b + 1], seeds[b:b + 1])
        assert np.array_equal(one[0], m[b]) and n1[0] == lines[b], b


def test_make_items_radial_layout():
    H, W = 64, 48
    items = ops.make_items(torch.rand(H, W, device=DEV), torch.tensor([0.0, 5.0], device=DEV), 3, radial=0.3)
    ref = synth.make_batch(2, H, W, "radial", 0.3, 5.0, seed0=3)
    for k, v in ref.items():
        assert items[k].shape == v.shape and items[k].dtype == torch.from_numpy(v).dtype and items[k].is_cuda, k
    for b in range(2):
        assert np.array_equal(items["mask"][b].cpu().numpy(), radial_mask(H, W, 0.3, 3 + b)[0])


@pytest.mark.parametrize("H,W", [(256, 256), (130, 130)])
def test_engine_reset_from_gt_equals_reset_of_make_items(H, W):
    B = 3
    params = O.init_unet_params(0, "default")
    den = UNetDenoiser2D(state_dict=params)
    gt = torch.rand(B, 1, H, W, device=DEV)
    a, b = PnPEngine(den, B, H, W, DEV), PnPEngine(den, B, H, W, DEV)
    a.reset_from_gt(gt, 10.0, 17, radial=0.3)
    b.reset(ops.make_items(gt, 10.0, 17, radial=0.3))
    names = ["x", "v", "z", "u", "y0", "mask", "gt"] + (["y0T", "maskT"] if a.prepared else [])
    for n in names:
        assert torch.equal(getattr(a, n), getattr(b, n)), n
    for k in range(B):
        assert np.array_equal(a.mask[k, 0].cpu().numpy(), radial_mask(H, W, 0.3, 17 + k)[0])
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
    with pytest.raises(ValueError):
        a.reset_from_gt(gt, 10.0, 17, accel=4, radial=0.3)


def test_rejection():
    H = W = 32
    fr = torch.full((2,), 0.3, dtype=torch.float64, device=DEV)
    seeds = torch.zeros(2, dtype=torch.int64, device=DEV)
    with pytest.raises(_lib.PnpError):
        ops.radial_masks(2, H, W, fr.cpu())
    with pytest.raises(_lib.PnpError):
        ops.radial_masks(2, H, W, fr, seeds.cpu())
    with pytest.raises(_lib.PnpError):
        ops.radial_masks(2, H, W, fr, out=torch.empty(2, H, W, dtype=torch.uint8))
    with pytest.raises(_lib.PnpError):
        ops.radial_masks(2, H, W, fr, lines_out=torch.empty(2, dtype=torch.int32))
    with pytest.raises(_lib.PnpError):
        ops.radial_masks(2, 1030, W, 0.3)
    with pytest.raises(_lib.PnpError):
        ops.radial_masks(2, H, 1, 0.3)
    with pytest.raises(TypeError):
        ops.radial_masks(2, H, W, fr.float())                       # a float32 frac could move the stop by a line
    with pytest.raises(ValueError):
        ops.make_items(torch.rand(2, H, W, device=DEV), 0.0, 0, accel=4, radial=0.3)
    lib = _lib.lib()
    out = torch.empty(2, H, W, dtype=torch.uint8, device=DEV)
    lines = torch.empty(2, dtype=torch.int32, device=DEV)
    st = _lib.stream_ptr()
    assert lib.pnp_radial_masks(fr.data_ptr(), 1, seeds.data_ptr(), out.data_ptr(), lines.data_ptr(), 2, H, W, st) == 0
    assert lib.pnp_radial_masks(fr.data_ptr(), 0, None, out.data_ptr(), None, 2, H, W, st) == 0
    for args in ((fr.data_ptr(), 1, seeds.data_ptr(), out.data_ptr(), out.data_ptr() + 8, 2, H, W, st),
                 (fr.data_ptr(), 1, seeds.data_ptr(), out.data_ptr(), lines.data_ptr(), 0, H, W, st),
                 (fr.data_ptr(), 1, out.data_ptr(), out.data_ptr(), lines.data_ptr(), 2, H, W, st)):
        assert lib.pnp_radial_masks(*args) < 0
        assert b"pnp_radial_masks" in lib.pnp_last_error()
    torch.cuda.synchronize()
