"""pnp_simulate_measurements / pnp_cartesian_masks (csrc/measure.cuh) through ops, PnPEngine.reset_from_gt and PnPEnv against
the float64 reference (tests/measure_reference.py): accuracy at radix and dense-DFT sizes, exact properties (mask zeros,
x0 = clamp(ATy0), determinism, batch-position independence), noise statistics, masks bit for bit, batches over 65535,
graph capture, the engine and env entry points, rejection."""
from collections import OrderedDict

import numpy as np
import pytest
import torch

from dt4image_restoration_b200 import _lib, ops, synth
from dt4image_restoration_b200.engine import PnPEngine
from dt4image_restoration_b200.env import PnPEnv
from dt4image_restoration_b200.noise import UNetDenoiser2D
from measure_reference import acs_cols, cartesian_mask, make_item, simulate
from oracle import pnp_oracle as O

pytestmark = pytest.mark.gpu
DEV = "cuda"
RADIX = [(32, 32), (64, 128), (128, 128), (256, 256), (256, 64), (512, 512)]
DENSE = [(2, 3), (45, 51), (130, 130), (136, 120), (1000, 37), (1024, 1024)]
SEEDS = [7, (1 << 40) + 3, -5]          # -5: an int64 seed is used as its uint64 bit pattern


def _tol(H, W):
    return (2e-6 if (H, W) in RADIX else 4e-6) * np.log2(H * W)


def _check_image(y0, x0, aty0, gt, mask, sigma, seed):
    """One image's outputs (complex64 [H, W], aty0 may be None) against the reference."""
    H, W = gt.shape
    r_y0, r_at, r_x0 = simulate(gt, mask, sigma, seed)
    t = _tol(H, W)
    assert np.abs(y0.cpu().numpy() - r_y0).max() <= t * np.abs(r_y0).max()
    assert np.abs(x0.cpu().numpy() - r_x0).max() <= 2 * t * np.abs(r_at).max()
    if aty0 is not None:
        assert np.abs(aty0.cpu().numpy() - r_at).max() <= 2 * t * np.abs(r_at).max()


def _inputs(B, H, W, seed, density=0.4):
    g = torch.Generator().manual_seed(seed)
    gt = torch.rand(B, 1, H, W, generator=g)
    mask = (torch.rand(B, H, W, generator=g) < density).to(torch.uint8)
    return gt, mask


@pytest.mark.parametrize("H,W", RADIX + DENSE)
def test_per_image_inputs_against_reference(H, W):
    B = 1 if H * W >= 512 * 512 else 3
    gt, mask = _inputs(B, H, W, H * 7 + W)
    sig = torch.tensor([0.0, 5.0, 15.0][:B])
    seeds = torch.tensor(SEEDS[:B], dtype=torch.int64)
    y0, x0, at = ops.simulate_measurements(gt.to(DEV), mask.to(DEV), sig.to(DEV), seeds.to(DEV))
    assert y0.shape == (B, 1, H, W) and y0.dtype == torch.complex64 and x0.shape == y0.shape and at.shape == y0.shape
    for b in range(B):
        _check_image(y0[b, 0], x0[b, 0], at[b, 0], gt[b, 0].numpy(), mask[b].numpy(), float(sig[b]), SEEDS[b])


@pytest.mark.parametrize("H,W", [(64, 128), (512, 512), (45, 51), (1024, 1024)])
def test_shared_gt_and_mask_scalar_sigma_no_aty0(H, W):
    gt, mask = _inputs(1, H, W, H + W)
    B = 2 if H * W >= 512 * 512 else 4
    y0, x0, at = ops.simulate_measurements(gt[0, 0].to(DEV), mask.to(DEV), 10.0, torch.arange(3, 3 + B, device=DEV),
                                           aty0=False)
    assert at is None and y0.shape == (B, 1, H, W)
    for b in (0, B - 1):
        _check_image(y0[b, 0], x0[b, 0], None, gt[0, 0].numpy(), mask[0].numpy(), 10.0, 3 + b)
    y1, x1, _ = ops.simulate_measurements(gt[0, 0].to(DEV), mask.to(DEV), 10.0, 3)   # int s0 = s0 + arange(B), B from mask
    assert torch.equal(y1[0], y0[0]) and torch.equal(x1[0], x0[0])


@pytest.mark.parametrize("H,W", [(128, 128), (45, 51)])
def test_exact_properties(H, W):
    gt, mask = _inputs(4, H, W, 3)
    y0, x0, at = ops.simulate_measurements(gt.to(DEV), mask.to(DEV), 15.0, 11)
    off = mask.to(DEV).reshape(4, 1, H, W) == 0
    assert torch.all(y0[off] == 0)
    assert torch.equal(torch.view_as_real(x0), torch.view_as_real(at).clamp(min=0))
    y0b, x0b, atb = ops.simulate_measurements(gt.to(DEV), mask.to(DEV), 15.0, 11)
    assert torch.equal(y0, y0b) and torch.equal(x0, x0b) and torch.equal(at, atb)


@pytest.mark.parametrize("H,W", [(256, 256), (130, 130)])
def test_batch_position_independence(H, W):
    B = 8
    gt, mask = _inputs(B, H, W, 5)
    sig = torch.linspace(0, 15, B)
    seeds = torch.arange(100, 100 + B, dtype=torch.int64)
    args = [t.to(DEV) for t in (gt, mask, sig, seeds)]
    y0, x0, at = ops.simulate_measurements(*args)
    perm = torch.randperm(B, generator=torch.Generator().manual_seed(1)).to(DEV)
    yp, xp, ap = ops.simulate_measurements(*[t[perm] for t in args])
    assert torch.equal(yp, y0[perm]) and torch.equal(xp, x0[perm]) and torch.equal(ap, at[perm])
    y1, _, _ = ops.simulate_measurements(*[t[5:6] for t in args])
    assert torch.equal(y1[0], y0[5])


@pytest.mark.parametrize("H,W", [(256, 256), (136, 120)])
def test_two_masks_agree_where_both_sample(H, W):
    gt, m1 = _inputs(2, H, W, 8, density=0.5)
    m2 = _inputs(2, H, W, 9, density=0.5)[1]
    ya, _, _ = ops.simulate_measurements(gt.to(DEV), m1.to(DEV), 10.0, 4)
    yb, _, _ = ops.simulate_measurements(gt.to(DEV), m2.to(DEV), 10.0, 4)
    both = ((m1 != 0) & (m2 != 0)).to(DEV).reshape(2, 1, H, W)
    assert both.sum() > 0 and torch.equal(ya[both], yb[both])


@pytest.mark.parametrize("B,H,W", [(2, 512, 512), (8, 1000, 37)])
def test_noise_statistics(B, H, W):
    gt = torch.zeros(B, 1, H, W, device=DEV)
    mask = torch.ones(1, H, W, dtype=torch.uint8, device=DEV)
    y0, _, _ = ops.simulate_measurements(gt, mask, 15.0, 21)
    n = torch.view_as_real(y0).double() * (255.0 / 15.0)
    nr, ni = n[..., 0].reshape(-1), n[..., 1].reshape(-1)
    for s in (nr, ni):
        assert abs(s.mean().item()) < 1e-2 and abs(s.var().item() - 1.0) < 2e-2
    assert abs(torch.corrcoef(torch.stack([nr, ni]))[0, 1].item()) < 1e-2


@pytest.mark.parametrize("H,W", [(256, 256), (45, 51), (2, 3), (1000, 37), (16, 1024)])
def test_cartesian_masks_match_reference(H, W):
    accel = [1, 2, 3, 4, 8, 16]
    seeds = [0, 1, 2, (1 << 33) + 5, -7, 1234567]
    got = ops.cartesian_masks(6, H, W, torch.tensor(accel, dtype=torch.int32, device=DEV),
                              torch.tensor(seeds, dtype=torch.int64, device=DEV)).cpu().numpy()
    for b in range(6):
        assert np.array_equal(got[b], cartesian_mask(H, W, accel[b], seeds[b], acs_cols(W))), b
    shared = ops.cartesian_masks(3, H, W, 4, 10).cpu().numpy()                # one accel, seeds 10, 11, 12
    for b in range(3):
        assert np.array_equal(shared[b], cartesian_mask(H, W, 4, 10 + b, acs_cols(W)))


def test_cartesian_masks_take_the_row_only_prox_path():
    H = W = 256
    mask = ops.cartesian_masks(4, H, W, 4, 0)
    y0, _, _ = ops.simulate_measurements(torch.rand(4, 1, H, W, device=DEV), mask, 10.0, 0)
    assert ops.ProxPrepared(y0, mask).column_only


@pytest.mark.parametrize("H,W", [(32, 32), (2, 3)])
def test_batch_over_65535(H, W):
    B = 65537
    g = torch.Generator(device=DEV).manual_seed(3)
    gt = torch.rand(B, 1, H, W, device=DEV, generator=g)
    mask = ops.cartesian_masks(B, H, W, 2, 0)
    sig = torch.rand(B, device=DEV, generator=g) * 15
    seeds = torch.arange(B, dtype=torch.int64, device=DEV) * 3
    y0, x0, at = ops.simulate_measurements(gt, mask, sig, seeds)
    for b in (0, 65535, B - 1):
        one = ops.simulate_measurements(gt[b:b + 1], mask[b:b + 1], sig[b:b + 1], seeds[b:b + 1])
        assert torch.equal(one[0][0], y0[b]) and torch.equal(one[1][0], x0[b]) and torch.equal(one[2][0], at[b])
        assert torch.equal(ops.cartesian_masks(1, H, W, 2, b)[0], mask[b])


@pytest.mark.parametrize("H,W", [(256, 256), (130, 130)])
def test_graph_capture(H, W):
    B = 3
    gt = torch.rand(B, 1, H, W, device=DEV)
    accel = torch.tensor([2, 4, 8], dtype=torch.int32, device=DEV)
    seeds = torch.tensor([5, 6, 7], dtype=torch.int64, device=DEV)
    sig = torch.tensor([0.0, 5.0, 10.0], device=DEV)
    mask = torch.empty(B, H, W, dtype=torch.uint8, device=DEV)
    outs = tuple(torch.empty(B, 1, H, W, dtype=torch.complex64, device=DEV) for _ in range(3))

    def body():
        ops.cartesian_masks(B, H, W, accel, seeds, out=mask)
        ops.simulate_measurements(gt, mask, sig, seeds, out=outs)

    body()
    eager = [mask.clone()] + [o.clone() for o in outs]
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        body()
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        body()
    mask.zero_()
    for o in outs:
        o.zero_()
    graph.replay()
    torch.cuda.synchronize()
    for a, b in zip(eager, [mask, *outs]):
        assert torch.equal(a, b)


@pytest.mark.parametrize("H,W,use_accel", [(64, 64, True), (130, 130, False)])
def test_engine_reset_from_gt_equals_reset_of_make_items(H, W, use_accel):
    B = 3
    params = O.init_unet_params(0, "default")
    den = UNetDenoiser2D(state_dict=params)
    gt = torch.rand(B, 1, H, W, device=DEV)
    kw = {"accel": 4} if use_accel else {"mask": torch.from_numpy(synth.radial_mask(H, W, 0.3)).to(DEV)}
    a, b = PnPEngine(den, B, H, W, DEV), PnPEngine(den, B, H, W, DEV)
    a.reset_from_gt(gt, 10.0, 17, **kw)
    b.reset(ops.make_items(gt, 10.0, 17, **kw))
    names = ["x", "v", "z", "u", "y0", "mask", "gt"] + (["y0T", "maskT"] if a.prepared else [])
    for n in names:
        assert torch.equal(getattr(a, n), getattr(b, n)), n
    for e in (a, b):
        e.set_actions(torch.tensor([0.1, 0.15, 0.2]), 0.5)
    for _ in range(3):
        a.step()
        b.step()
    for n in ("x", "z", "u", "v"):
        assert torch.equal(getattr(a, n), getattr(b, n)), n


def test_make_items_layout():
    H, W = 64, 48
    items = ops.make_items(torch.rand(H, W, device=DEV), torch.tensor([0.0, 5.0], device=DEV), 3, accel=4)
    ref = synth.make_batch(2, H, W, "cartesian", 4, 5.0, seed0=3)
    for k, v in ref.items():
        assert items[k].shape == v.shape and items[k].dtype == torch.from_numpy(v).dtype and items[k].is_cuda, k


@pytest.mark.parametrize("H,W,kind,sigma", [(256, 256, "cartesian", 10.0), (130, 130, "radial", 5.0)])
def test_env_against_oracle(H, W, kind, sigma):
    seed = 4
    params = O.init_unet_params(0, "default")
    gt = synth.phantom(H, W, seed)
    if kind == "cartesian":
        items = ops.make_items(torch.from_numpy(gt).to(DEV), sigma, seed, accel=4)
        mask = cartesian_mask(H, W, 4, seed, acs_cols(W))
    else:
        mask = synth.radial_mask(H, W, 0.3)
        items = ops.make_items(torch.from_numpy(gt).to(DEV), sigma, seed, mask=torch.from_numpy(mask).to(DEV))
    assert np.array_equal(items["mask"].cpu().numpy()[0], mask)
    ref_item = make_item(gt, mask, sigma, seed)
    env = PnPEnv(30, UNetDenoiser2D(state_dict=params), DEV)
    st = env.reset(items, DEV)
    ref = O.reset(ref_item)
    assert (st["z"].cpu() - ref["z"]).abs().max() < 1e-3
    for k in range(3):
        action = OrderedDict({"T": torch.zeros(1, device=DEV), "mu": torch.tensor([0.3 + 0.2 * k], device=DEV),
                              "sigma_d": torch.tensor([0.1], device=DEV)})
        st, _ = env.step(st, action)
        ref, _ = O.step(params, ref, {k2: v.cpu() for k2, v in action.items()})
        assert (st["x"].cpu() - ref["x"]).abs().max() < 1e-3, k
    assert (st["z"].cpu() - ref["z"]).abs().max() < 1e-3 and (st["u"].cpu() - ref["u"]).abs().max() < 1e-3


def test_rejection():
    lib = _lib.lib()
    H = W = 32
    gt = torch.rand(2, H, W, device=DEV)
    mask = torch.ones(2, H, W, dtype=torch.uint8, device=DEV)
    sig = torch.zeros(1, device=DEV)
    seeds = torch.zeros(2, dtype=torch.int64, device=DEV)
    y0, x0, at = (torch.empty(2, H, W, dtype=torch.complex64, device=DEV) for _ in range(3))
    st = _lib.stream_ptr()

    def sim(**kw):
        a = dict(gt=gt.data_ptr(), gs=H * W, mask=mask.data_ptr(), ms=H * W, sig=sig.data_ptr(), ss=0,
                 seeds=seeds.data_ptr(), y0=y0.data_ptr(), x0=x0.data_ptr(), at=at.data_ptr(), B=2, H=H, W=W)
        a.update(kw)
        return lib.pnp_simulate_measurements(a["gt"], a["gs"], a["mask"], a["ms"], a["sig"], a["ss"], a["seeds"], a["y0"],
                                             a["x0"], a["at"], a["B"], a["H"], a["W"], st)

    assert sim() == 0 and sim(at=None) == 0
    for kw in ({"gt": None}, {"mask": None}, {"sig": None}, {"seeds": None}, {"y0": None}, {"x0": None}, {"B": 0},
               {"H": 1}, {"W": 1025}, {"ms": -1}, {"y0": gt.data_ptr()}, {"x0": mask.data_ptr()}, {"at": y0.data_ptr()},
               {"x0": y0.data_ptr() + 8}):
        assert sim(**kw) < 0, kw
        assert b"pnp_simulate_measurements" in lib.pnp_last_error()
    acc = torch.full((1,), 4, dtype=torch.int32, device=DEV)
    out = torch.empty(2, H, W, dtype=torch.uint8, device=DEV)

    def masks(**kw):
        a = dict(acc=acc.data_ptr(), ast=0, seeds=seeds.data_ptr(), acs=3, out=out.data_ptr(), B=2, H=H, W=W)
        a.update(kw)
        return lib.pnp_cartesian_masks(a["acc"], a["ast"], a["seeds"], a["acs"], a["out"], a["B"], a["H"], a["W"], st)

    assert masks() == 0
    for kw in ({"acc": None}, {"seeds": None}, {"out": None}, {"acs": 0}, {"B": 0}, {"H": 1}, {"W": 1025}):
        assert masks(**kw) < 0, kw
        assert b"pnp_cartesian_masks" in lib.pnp_last_error()
    with pytest.raises(_lib.PnpError):
        ops.simulate_measurements(torch.rand(2, H, W), mask, 0.0, 0)
    with pytest.raises(_lib.PnpError):
        ops.simulate_measurements(gt, mask.cpu(), 0.0, 0)
    with pytest.raises(_lib.PnpError):
        ops.simulate_measurements(gt, mask, 0.0, seeds.cpu())
    with pytest.raises(_lib.PnpError):
        ops.cartesian_masks(2, H, W, acc.cpu(), 0)
    with pytest.raises(_lib.PnpError):
        ops.simulate_measurements(torch.rand(2, 1, 1, 1030, device=DEV), torch.ones(1, 1, 1030, dtype=torch.uint8,
                                                                                    device=DEV), 0.0, 0)
    with pytest.raises(ValueError):
        ops.make_items(gt, 0.0, 0)
    torch.cuda.synchronize()
