"""``ops.ProxPrepared`` refilled in place (``empty`` + ``prepare``), as the engine and the graphed env step use it: the
buffers keep their addresses, and every result equals that of a freshly built ``ProxPrepared``.  Needs a B200."""
import pytest
import torch

from dt4image_restoration_b200 import ops

pytestmark = pytest.mark.gpu
DEV = "cuda"
B = 3


def trajectory(H, W, kind, seed):
    """(y0, mask) of a seeded batch: Cartesian 4x (column-only masks) or radial 30 % (general masks)."""
    gt = torch.rand(B, 1, H, W, generator=torch.Generator(DEV).manual_seed(seed), device=DEV)
    kw = {"accel": 4} if kind == "cartesian" else {"radial": 0.3}
    it = ops.make_items(gt, 5.0, seed, **kw)
    return torch.view_as_complex(it["y0"]), it["mask"]


def prox_results(prep, H, W):
    g = torch.Generator(DEV).manual_seed(5)
    x = torch.rand(B, 1, H, W, generator=g, device=DEV)
    u = torch.randn(B, 1, H, W, dtype=torch.complex64, generator=g, device=DEV) * 0.1
    mu = torch.tensor([0.2, 0.5, 0.8], device=DEV)
    return [t for kind in (-1, None) for t in prep.prox_dual(x, u, mu, kind=kind)]


@pytest.mark.parametrize("H,W", [(256, 256), (128, 128), (64, 64)])
def test_empty_before_prepare(H, W):
    prep = ops.ProxPrepared.empty(B, H, W, DEV)
    assert prep.probe.get() == -1
    assert prep.launches == {256: 2, 128: 1, 64: 4}[H]       # the both-kernels launch while the kind is unknown
    assert not prep.y0p.any() and not prep.maskp.any()


@pytest.mark.parametrize("H,W", [(256, 256), (128, 128), (64, 64)])
@pytest.mark.parametrize("first,second", [("cartesian", "cartesian"), ("radial", "radial"),
                                          ("radial", "cartesian"), ("cartesian", "radial")])
def test_prepare_in_place_equals_fresh(H, W, first, second):
    prep = ops.ProxPrepared.empty(B, H, W, DEV)
    ptrs = (prep.y0p.data_ptr(), prep.maskp.data_ptr())
    prep.prepare(*trajectory(H, W, first, 1))
    y0, mask = trajectory(H, W, second, 2)
    prep.prepare(y0, mask)
    fresh = ops.ProxPrepared(y0, mask)
    assert (prep.y0p.data_ptr(), prep.maskp.data_ptr()) == ptrs
    assert prep.column_only == fresh.column_only == (second == "cartesian")
    assert prep.probe.get() == fresh.probe.get() >= 0 and prep.launches == fresh.launches
    if first == second:
        # a change of mask kind leaves the regions the new kind never reads as they were, so only the same kind gives
        # byte-equal buffers
        assert torch.equal(prep.y0p, fresh.y0p) and torch.equal(prep.maskp, fresh.maskp)
    for a, b in zip(prox_results(prep, H, W), prox_results(fresh, H, W)):
        assert torch.equal(a, b)
