"""CPU self-test of the per-launch denoiser references (tests/unet_launch_reference.py), no GPU needed.

1. Composed in float64, the launch references reproduce the oracle's U-Net (pinned to the reference's own outputs): pad
   offsets, align_corners, concat order and the residual are restated right.
2. The bounds accept what a correct kernel may return: the bf16 rounding of the exact result, and an fp32 recomputation
   with another summation order.
3. The bounds reject small, realistic kernel bugs on the oracle's own activations (kaiming weights, seed 1), so they cannot
   be loosened until such a bug passes.
"""
import functools

import pytest
import torch
import torch.nn.functional as F

from oracle import pnp_oracle as O
import unet_launch_reference as R

BLOCKS = ("inc", "down1", "down2", "down3", "down4", "up1", "up2", "up3", "up4")


def wb(params, block, i):
    p = f"{O._block_prefix(block)}.conv-{i}.conv2d"
    return params[p + ".weight"], params[p + ".bias"]


def compose(params, v, sigma):
    """The plan's launches chained in float64 with un-rounded weights and activations -> preclamp [B,H,W]."""
    x = R.first_conv(v, sigma, *wb(params, "inc", 0))[0]
    for i in (1, 2):
        x = R.conv3x3(x, None, *wb(params, "inc", i))[0]
    skips = [x]
    for blk in BLOCKS[1:5]:
        x = R.maxpool(x)
        for i in range(3):
            x = R.conv3x3(x, None, *wb(params, blk, i))[0]
        skips.append(x)
    x = skips.pop()
    for blk in BLOCKS[5:]:
        skip = skips.pop()
        up = R.upsample(x, skip.shape[1], skip.shape[2])[0]
        x = R.conv3x3(skip, up, *wb(params, blk, 0))[0]
        for i in (1, 2) if blk != "up4" else (1,):
            x = R.conv3x3(x, None, *wb(params, blk, i))[0]
    return R.final(x, *wb(params, "up4", 2), params["outc.conv.weight"], params["outc.conv.bias"], v)[0]


@pytest.mark.parametrize("B,H,W", [(1, 45, 51), (2, 64, 64), (2, 31, 17)])
@pytest.mark.parametrize("kind", ["default", "kaiming"])
def test_composed_references_reproduce_the_oracle(B, H, W, kind):
    params = O.init_unet_params(1, kind)
    g = torch.Generator().manual_seed(H * W)
    v = torch.rand(B, 1, H, W, generator=g)
    sigma = torch.rand(B, generator=g) * 0.2 + 0.02
    got = compose(params, v[:, 0], sigma)
    ref32 = O.denoise(params, v, sigma, clamp=False)[:, 0]
    ref64 = O.denoise({k: t.double() for k, t in params.items()}, v.double(), sigma.double(), clamp=False)[:, 0]
    # same semantics: float64 agrees with float64 to rounding; the pinned fp32 oracle to fp32 noise
    assert (got - ref64).abs().max() < 1e-10
    assert (got - ref32.double()).abs().max() < 1e-4


# ------------------------------------------------------------------------------------------------
# oracle activations as the GPU would hold them (bf16 NHWC)
# ------------------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def taps(B, H, W, depth="all"):
    params = O.init_unet_params(1, "kaiming")
    g = torch.Generator().manual_seed(H + W)
    v = torch.rand(B, 1, H, W, generator=g)
    sigma = torch.rand(B, generator=g) * 0.2 + 0.02
    t = {}
    if depth == "inc":              # large sizes: only the first block
        x = torch.cat([v, torch.ones(B, 1, H, W) * sigma.view(B, 1, 1, 1)], dim=1)
        O._conv_block(params, O._block_prefix("inc"), x, t, "inc")
    else:
        O.denoise(params, v, sigma, clamp=False, taps=t)
    act = {k: R.nhwc(x).to(torch.bfloat16) for k, x in t.items() if x.dim() == 4}
    return params, v[:, 0], sigma, act


def bf16_of_fp32_conv(x, w, b, reorder=True):
    """A correct tensor-core conv as fp32 arithmetic can give it: fp32 conv with the input channels in reverse order (another
    summation order), bias, LeakyReLU, rounded to bf16."""
    xx = R.nchw(x).float()
    ww = w.float()
    if reorder:
        xx, ww = xx.flip(1), ww.flip(1)
    y = F.leaky_relu(F.conv2d(xx, ww, b.float(), padding=1), R.SLOPE)
    return R.nhwc(y).to(torch.bfloat16)


def rejects(got, ref, bound):
    return R.compare(got, ref, bound)[2] > 0


CONV_CASES = [
    # (B, H, W, block, conv index, taps depth): the tile / channel structure of the plan's convs
    (1, 256, 256, "inc", 2, "inc"),        # the benchmark size (the mutations the chain-level test lets through)
    (2, 64, 64, "inc", 1, "all"),
    (2, 31, 17, "down1", 1, "all"),
    (1, 45, 51, "down2", 2, "all"),
    (1, 45, 51, "up3", 0, "all"),          # concat of skip and upsampled tensors
    (2, 64, 64, "up2", 1, "all"),
]


def conv_case(B, H, W, block, i, depth):
    params, _, _, act = taps(B, H, W, depth)
    w, b = wb(params, block, i)
    wq = R.bf16r(w)
    if block.startswith("up") and i == 0:
        lvl = {"up1": 3, "up2": 2, "up3": 1, "up4": 0}[block]
        src = {3: "down3", 2: "down2", 1: "down1", 0: "inc"}[lvl]
        in0, in1 = act[f"{src}.conv-2"], act[f"{block}.upsampled"]
    elif i == 0:
        in0, in1 = act[f"{block}.pooled"], None
    else:
        in0, in1 = act[f"{block}.conv-{i - 1}"], None
    return in0, in1, wq, b


@pytest.mark.parametrize("case", CONV_CASES, ids=lambda c: f"{c[0]}x{c[1]}x{c[2]}-{c[3]}.conv-{c[4]}")
def test_conv_bound_accepts_rounding_and_rejects_mutations(case):
    in0, in1, wq, b = conv_case(*case)
    ref, bound = R.conv3x3(in0, in1, wq, b)
    x = in0 if in1 is None else torch.cat([in0, in1], dim=-1)
    assert not rejects(ref.to(torch.bfloat16), ref, bound)
    good = bf16_of_fp32_conv(x, wq, b)
    assert not rejects(good, ref, bound), R.compare(good, ref, bound)
    B, H, W, C = good.shape
    ty, tx = (H // 16) // 2, (W // 16) // 2          # a tile in the middle
    ys, xs = slice(16 * ty, 16 * ty + 16), slice(16 * tx, 16 * tx + 16)
    # one 16-pixel row of one tile zeroed
    m = good.clone(); m[0, 16 * ty + 5, xs, :] = 0
    assert rejects(m, ref, bound)
    # one tile 1 % off
    m = good.clone(); m[0, ys, xs, :] = (m[0, ys, xs, :].double() * 1.01).to(torch.bfloat16)
    assert rejects(m, ref, bound)
    # two neighbouring tiles swapped (a wrong tile decode), over the region they have in common
    tiles = [(i, y, x) for i in range(B) for y in range(0, H, 16) for x in range(0, W, 16)]
    if len(tiles) > 1:
        (i1, y1, x1), (i2, y2, x2) = tiles[len(tiles) // 2 - 1], tiles[len(tiles) // 2]
        h, w = min(16, H - y1, H - y2), min(16, W - x1, W - x2)
        m = good.clone()
        m[i1, y1:y1 + h, x1:x1 + w], m[i2, y2:y2 + h, x2:x2 + w] = good[i2, y2:y2 + h, x2:x2 + w], good[i1, y1:y1 + h, x1:x1 + w]
        assert rejects(m, ref, bound)
    # one 3x3 tap of one 32-channel slice missing
    wm = wq.clone(); wm[:, -32:, 2, 0] = 0
    assert rejects(bf16_of_fp32_conv(x, wm, b, reorder=False), ref, bound)
    # the bias of one channel dropped (the channel whose bias has the median magnitude)
    c = int(b.abs().argsort()[len(b) // 2])
    bm = b.clone(); bm[c] = 0
    assert rejects(bf16_of_fp32_conv(x, wq, bm, reorder=False), ref, bound)


@pytest.mark.parametrize("B,H,W", [(2, 31, 17), (1, 45, 51), (2, 64, 64)])
def test_first_conv_bound(B, H, W):
    params, v, sigma, _ = taps(B, H, W)
    w, b = wb(params, "inc", 0)
    ref, bound = R.first_conv(v, sigma, w, b)
    x = torch.stack([v, sigma.view(B, 1, 1).expand(B, H, W)], dim=1)
    good = R.nhwc(F.leaky_relu(F.conv2d(x.flip(1), w.flip(1), b, padding=1), R.SLOPE)).to(torch.bfloat16)
    assert not rejects(good, ref, bound)
    # the sigma channel padded with sigma instead of zero (a wrong edge case of the pre-summed taps)
    xp = torch.cat([F.pad(v[:, None], (1, 1, 1, 1)), F.pad(x[:, 1:], (1, 1, 1, 1), mode="replicate")], dim=1)
    bad = R.nhwc(F.leaky_relu(F.conv2d(xp, w, b), R.SLOPE)).to(torch.bfloat16)
    assert rejects(bad, ref, bound)
    # the last row of an odd-H image left out (the row pair's second row)
    m = good.clone(); m[:, H - 1] = 0
    assert rejects(m, ref, bound)


@pytest.mark.parametrize("B,H,W", [(2, 31, 17), (2, 45, 51)])
def test_pool_is_exact_and_rejects_the_out_of_image_row(B, H, W):
    """At odd H the last row is dropped by MaxPool2d(2) (floor mode).  A pool that takes it writes pooled row Hp of image 0,
    which is row 0 of image 1 in the [B, Hp, Wp, C] buffer; likewise at odd W column Wp of a row is column 0 of the next."""
    _, _, _, act = taps(B, H, W)
    out = act["inc.conv-2"]
    ref = R.maxpool(out)
    exact = torch.zeros_like(ref)
    assert R.compare(act["down1.pooled"], ref, exact)[0] == 0.0
    Hp, Wp, C = H // 2, W // 2, ref.shape[-1]
    assert H % 2 == 1 and W % 2 == 1
    # the out-of-image row / column counts as 0 (what the zero-padded conv input would leave after a ReLU-like max)
    last_row = torch.maximum(out[0, H - 1, 0:2 * Wp:2], out[0, H - 1, 1:2 * Wp:2]).clamp_min(0)
    m = ref.clone().reshape(-1, C)
    m[Hp * Wp:Hp * Wp + Wp] = last_row.double()
    assert rejects(m.reshape(ref.shape), ref, exact)
    last_col = torch.maximum(out[0, 0:2 * Hp:2, W - 1], out[0, 1:2 * Hp:2, W - 1]).clamp_min(0)
    m = ref.clone().reshape(B * Hp, Wp, C)
    m[1:Hp, 0] = last_col[:Hp - 1].double()          # row r's column Wp is row r + 1's column 0
    assert rejects(m.reshape(ref.shape), ref, exact)


@pytest.mark.parametrize("B,H,W,block", [(1, 45, 51, "up4"), (1, 45, 51, "up3"), (1, 45, 51, "up2"), (2, 31, 17, "up4"),
                                         (2, 31, 17, "up1"), (2, 64, 64, "up4")])
def test_upsample_bound(B, H, W, block):
    _, _, _, act = taps(B, H, W)
    lvl = {"up1": 3, "up2": 2, "up3": 1, "up4": 0}[block]
    low = act["down4.conv-2"] if lvl == 3 else act[f"{BLOCKS[5 + (3 - lvl) - 1]}.conv-2"]
    Ho, Wo = H >> lvl, W >> lvl
    ref, bound, inside = R.upsample(low, Ho, Wo)
    assert bool((ref[:, ~inside] == 0).all()) and bool((bound[:, ~inside] == 0).all())
    up = F.interpolate(R.nchw(low).float(), scale_factor=2, mode="bilinear", align_corners=True)
    dy, dx = Ho - up.shape[2], Wo - up.shape[3]
    # torch's fp32 upsample (the oracle's operation), padded and rounded to bf16, is accepted
    good = R.nhwc(F.pad(up, (dx // 2, dx - dx // 2, dy // 2, dy - dy // 2))).to(torch.bfloat16)
    assert not rejects(good, ref, bound), R.compare(good, ref, bound)
    # align_corners=False (the same thing for a 1x1 source)
    bad = F.interpolate(R.nchw(low).float(), scale_factor=2, mode="bilinear", align_corners=False)
    assert low.shape[1:3] == (1, 1) or rejects(R.nhwc(F.pad(bad, (dx // 2, dx - dx // 2, dy // 2, dy - dy // 2))).to(torch.bfloat16), ref, bound)
    # the pad split swapped: the larger half on the leading side
    if dx % 2 or dy % 2:
        bad = F.pad(up, (dx - dx // 2, dx // 2, dy - dy // 2, dy // 2))
        assert rejects(R.nhwc(bad).to(torch.bfloat16), ref, bound)


def test_upsample_bound_covers_fp32_weights_at_large_sizes():
    """The fp32 interpolation weights err by up to 2^-23 h at source size h: an fp32 upsample 256 -> 512 stays inside."""
    g = torch.Generator().manual_seed(5)
    x = (torch.randn(1, 256, 256, 8, generator=g) * 4).to(torch.bfloat16)
    ref, bound, _ = R.upsample(x, 512, 512)
    got = R.nhwc(F.interpolate(R.nchw(x).float(), scale_factor=2, mode="bilinear", align_corners=True)).to(torch.bfloat16)
    assert not rejects(got, ref, bound), R.compare(got, ref, bound)


@pytest.mark.parametrize("B,H,W,kind", [(2, 31, 17, "kaiming"), (1, 45, 51, "kaiming"), (2, 64, 64, "default")])
def test_final_bound(B, H, W, kind):
    params = O.init_unet_params(1, kind)
    _, v, sigma, _ = taps(B, H, W)
    t = {}
    O.denoise(params, v[:, None], sigma, clamp=False, taps=t)
    x = R.nhwc(t["up4.conv-1"]).to(torch.bfloat16)
    w, b = wb(params, "up4", 2)
    wq = R.bf16r(w)
    wout, bout = params["outc.conv.weight"].reshape(-1), params["outc.conv.bias"]
    ref, bound = R.final(x, wq, b, wout, bout, v)
    # fp32 recomputation with the channels reordered
    a = F.leaky_relu(F.conv2d(R.nchw(x).float().flip(1), wq.float().flip(1), b, padding=1), R.SLOPE)
    good = v + (a * wout.view(1, -1, 1, 1)).sum(1) + bout
    assert not rejects(good, ref, bound), R.compare(good, ref, bound)
    assert rejects(good - bout, ref, bound)           # FINAL without bout
