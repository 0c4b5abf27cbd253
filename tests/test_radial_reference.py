"""The float64 radial-mask reference (tests/radial_reference.py) on its own, and pnp_radial_masks' C-ABI without a GPU."""
import math

import numpy as np
import pytest

from dt4image_restoration_b200 import _lib, synth
from radial_reference import half_length, phi, radial_mask

SHAPES = [(2, 3), (3, 2), (16, 16), (30, 34), (45, 51), (64, 48), (128, 128), (130, 130), (136, 120), (256, 256),
          (512, 512), (1000, 1000), (1024, 1024), (1024, 37)]
FRACS = [0.05, 0.1, 0.2, 0.3, 0.5, 0.9, 1.0]


@pytest.mark.parametrize("H,W", SHAPES)
def test_unseeded_reference_equals_synth_radial_mask(H, W):
    fracs = FRACS + [0.0, -0.5, float("nan")] + ([1.5] if H * W <= 512 * 512 else [])
    for f in fracs:
        m, n = radial_mask(H, W, f)
        assert m.dtype == np.uint8 and m.shape == (H, W)
        assert np.array_equal(m, synth.radial_mask(H, W, f)), f
        if not f > 0:                                   # frac <= 0 or NaN: no line
            assert n == 0 and not m.any(), f
        if f > 1:                                       # never reached: runs to the line cap
            assert n == 8 * max(H, W), f


def test_half_length_matches_synth_formula_at_every_size():
    H, W = np.meshgrid(np.arange(2, 1025), np.arange(2, 1025), indexing="ij")
    s = H * H + W * W
    r = np.floor(np.sqrt(s) / 2).astype(np.int64)
    for _ in range(2):
        r += 4 * r * r < s
    assert np.all(4 * r * r >= s) and np.all(4 * (r - 1) * (r - 1) < s)
    assert np.array_equal(r + 1, np.ceil(np.hypot(H, W) / 2).astype(np.int64) + 1)
    for (h, w) in SHAPES:
        assert half_length(h, w) == int(r[h - 2, w - 2]) + 1


def _nudged(ks: int, kc: int):
    """sin / cos moved by |ks| / |kc| ulp (sign = direction)."""
    def sincos(ang):
        s, c = np.sin(ang), np.cos(ang)
        for _ in range(abs(ks)):
            s = np.nextafter(s, np.inf if ks > 0 else -np.inf)
        for _ in range(abs(kc)):
            c = np.nextafter(c, np.inf if kc > 0 else -np.inf)
        return s, c
    return sincos


@pytest.mark.parametrize("H,W", [(2, 3), (3, 2), (30, 34), (45, 51), (64, 48), (130, 130), (136, 120), (256, 256)])
def test_masks_do_not_change_when_sin_cos_move_by_3_ulp(H, W):
    """Device and host sin / cos need not agree to the last bit; the masks must not depend on that."""
    for f in (0.05, 0.2, 0.3, 0.5, 1.0):
        for seed in (None, 11):
            ref, n = radial_mask(H, W, f, seed)
            for ks, kc in ((3, -3), (-3, 3), (3, 3), (-3, -3), (1, -1), (-1, 1)):
                m, _ = radial_mask(H, W, f, seed, sincos=_nudged(ks, kc))
                assert np.array_equal(m, ref), (f, seed, ks, kc)


def test_phi_in_zero_pi():
    assert phi(None) == 0.0
    ph = [phi(s) for s in range(2000)] + [phi((1 << 63) + s) for s in range(50)]
    assert all(0.0 <= p < math.pi for p in ph)
    assert float(np.float64(0xFFFFFFFF) * (np.pi * 2.0 ** -32)) < math.pi     # the largest Philox word
    assert max(ph) > 3.0 and min(ph) < 0.1 and len(set(ph)) == len(ph)


def test_distinct_seeds_give_distinct_masks():
    masks = [radial_mask(256, 256, 0.3, s)[0] for s in range(8)]
    for i in range(8):
        for j in range(i):
            assert not np.array_equal(masks[i], masks[j]), (i, j)
    assert not np.array_equal(masks[0], radial_mask(256, 256, 0.3)[0])


def test_negative_seed_is_its_uint64_bit_pattern():
    a = radial_mask(256, 256, 0.3, -5)
    b = radial_mask(256, 256, 0.3, (1 << 64) - 5)
    assert np.array_equal(a[0], b[0]) and a[1] == b[1]


@pytest.mark.parametrize("H,W", [(16, 16), (45, 51), (256, 256), (1024, 37)])
def test_line_count_is_minimal(H, W):
    for f in (0.05, 0.3, 0.9, 1.0, 1.5):
        for seed in (None, 3):
            m, n = radial_mask(H, W, f, seed)
            target = f * H * W
            assert int(m.sum()) >= target or n == 8 * max(H, W)
            if n < 8 * max(H, W):
                before = radial_mask(H, W, f, seed, max_lines=n - 1)[0]
                assert int(before.sum()) < target, (f, seed)


@pytest.mark.parametrize("H,W", [(2, 3), (3, 2), (45, 51), (256, 256)])
def test_centre_pixel_is_set_when_a_line_is_drawn(H, W):
    for f in (1e-9, 0.05, 0.3):
        for seed in (None, 1, -9):
            m, n = radial_mask(H, W, f, seed)
            assert n >= 1 and m[H // 2, W // 2] == 1


def test_c_abi_rejects_bad_arguments_without_a_gpu():
    """Argument checks run before the init check, so they answer on a machine without a GPU (fake addresses are never
    dereferenced: every call below is refused)."""
    lib = _lib.load()
    F, S, M, L = 1 << 20, 1 << 24, 1 << 30, 1 << 32                  # frac, seeds, mask_out (2 x 64x64 bytes), lines_out

    def masks(frac=F, st=1, seeds=S, out=M, lines=L, B=2, H=64, W=64):
        return lib.pnp_radial_masks(frac, st, seeds, out, lines, B, H, W, None)

    for kw in ({"frac": None}, {"out": None}, {"B": 0}, {"B": -3}, {"st": -1}, {"H": 1}, {"W": 1025}, {"H": 2000},
               {"lines": M + 4096}, {"lines": M + 2 * 64 * 64 - 4}, {"lines": M - 4}, {"out": L - 100},
               {"frac": M + 8}, {"seeds": M}, {"seeds": L + 4}):
        assert masks(**kw) < 0, kw
        assert b"pnp_radial_masks" in lib.pnp_last_error(), kw


def test_call_before_init_fails_with_a_message():
    lib = _lib.load()
    if _lib._inited:
        pytest.skip("the library was initialised by an earlier test in this process")
    assert lib.pnp_radial_masks(1 << 20, 0, None, 1 << 30, None, 1, 8, 8, None) < 0
    assert b"pnp_init" in lib.pnp_last_error()
