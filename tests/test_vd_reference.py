"""The float64 variable-density mask reference (tests/vd_reference.py) on its own, and pnp_variable_density_masks' C-ABI
without a GPU."""
import numpy as np
import pytest

from dt4image_restoration_b200 import _lib
from vd_reference import acs_block, acs_size, density, keys, n_keep, uniforms, vd_mask

SHAPES = [(2, 3), (3, 2), (45, 51), (256, 256), (1024, 37)]
ACCELS = [1, 2, 3, 4, 8, 0, -3]
TIE_SEEDS = [533, 1284]                 # 256^2, accel 2, power 0, 20x20 ACS: two equal float keys straddle the threshold


def _acs_cases(H, W):
    return [(0, 0), (1, 1), (H, W), (H, W - W // 3), (acs_size(H), acs_size(W))]     # (H, W - W//3): |ACS| > n_keep


@pytest.mark.parametrize("H,W", SHAPES)
def test_count_and_acs(H, W):
    for accel in ACCELS:
        for ah, aw in _acs_cases(H, W):
            m = vd_mask(H, W, accel, 7, 3, ah, aw)
            acs = acs_block(H, W, ah, aw)
            assert m.dtype == np.uint8 and m.shape == (H, W)
            assert int(acs.sum()) == ah * aw and m[acs].all(), (accel, ah, aw)
            assert int(m.sum()) == max(n_keep(H, W, accel), ah * aw), (accel, ah, aw)


def test_n_keep_rule():
    assert n_keep(256, 256, 4) == 16384 and n_keep(45, 51, 8) == 286 and n_keep(2, 3, 8) == 1
    assert n_keep(45, 51, 1) == n_keep(45, 51, 0) == n_keep(45, 51, -3) == 45 * 51


@pytest.mark.parametrize("H,W", [(2, 3), (45, 51), (256, 256)])
def test_power_zero_key_is_u(H, W):
    for seed in (0, 5, -2):
        assert np.array_equal(keys(H, W, seed, 0), uniforms(H, W, seed).astype(np.float32))


@pytest.mark.parametrize("H,W", SHAPES + [(64, 48), (3, 3)])
def test_zero_density_only_at_the_corners_and_taken_last(H, W):
    cy, cx = H // 2, W // 2
    ky = (np.arange(H) - cy) / cy
    kx = (np.arange(W) - cx) / cx
    corner = (np.abs(ky)[:, None] == 1) & (np.abs(kx)[None, :] == 1)
    for power in (1, 3, 16):
        w, r = density(H, W, power)
        assert np.array_equal(w == 0, corner) and np.array_equal(r == 1, corner)
        assert np.all((r >= 0) & (r <= 1))
        k = keys(H, W, 3, power)
        assert np.all(np.isinf(k[corner])) and np.all(k[~corner] > 0)
        # the corners are sampled only when nothing else is left
        assert n_keep(H, W, 2) <= H * W - int(corner.sum())
        assert not vd_mask(H, W, 2, 3, power, 0, 0)[corner].any() and vd_mask(H, W, 1, 3, power, 0, 0).all()


@pytest.mark.parametrize("power", [1, 3, 8])
def test_density_falls_with_radius(power):
    H = W = 256
    cy, cx = H // 2, W // 2
    rr = np.sqrt(0.5 * (((np.arange(H) - cy) / cy)[:, None] ** 2 + ((np.arange(W) - cx) / cx)[None, :] ** 2))
    dens = np.zeros(5)
    for seed in range(3):
        m = vd_mask(H, W, 4, seed, power, 0, 0)
        dens += [m[(rr >= lo) & (rr < lo + 0.2)].mean() for lo in np.arange(0.0, 1.0, 0.2)]
    assert np.all(np.diff(dens) < 0), dens


def test_power_zero_is_uniform():
    H = W = 256
    cy, cx = H // 2, W // 2
    rr = np.sqrt(0.5 * (((np.arange(H) - cy) / cy)[:, None] ** 2 + ((np.arange(W) - cx) / cx)[None, :] ** 2))
    m = vd_mask(H, W, 4, 1, 0, 0, 0)
    dens = np.array([m[(rr >= lo) & (rr < lo + 0.2)].mean() for lo in np.arange(0.0, 1.0, 0.2)])
    assert np.all(np.abs(dens - 0.25) < 0.02), dens


@pytest.mark.parametrize("seed", TIE_SEEDS)
def test_straddling_tie_goes_to_the_smaller_p(seed):
    H = W = 256
    a = acs_size(H)
    assert a == 20
    acs = acs_block(H, W, a, a).reshape(-1)
    m = vd_mask(H, W, 2, seed, 0, a, a).reshape(-1)
    k = keys(H, W, seed, 0).reshape(-1)
    threshold = k[m.astype(bool) & ~acs].max()
    tied = np.flatnonzero((k == threshold) & ~acs)
    taken = tied[m[tied] == 1]
    left = tied[m[tied] == 0]
    assert taken.size >= 1 and left.size >= 1, tied          # the tie straddles the threshold
    assert taken.max() < left.min()
    assert np.all(k[~acs & (m == 0)] >= threshold)


def test_distinct_seeds_give_distinct_masks():
    masks = [vd_mask(64, 64, 4, s, 3, 5, 5) for s in range(6)]
    for i in range(6):
        for j in range(i):
            assert not np.array_equal(masks[i], masks[j]), (i, j)
    assert np.array_equal(vd_mask(64, 64, 4, -5, 3, 5, 5), vd_mask(64, 64, 4, (1 << 64) - 5, 3, 5, 5))


def test_c_abi_rejects_bad_arguments_without_a_gpu():
    """Argument checks run before the init check, so they answer on a machine without a GPU (fake addresses are never
    dereferenced: every call below is refused)."""
    lib = _lib.load()
    A, S, M = 1 << 20, 1 << 24, 1 << 30                   # accel, seeds, mask_out (2 x 64x64 bytes)

    def masks(accel=A, st=1, seeds=S, ah=5, aw=5, power=3, out=M, B=2, H=64, W=64):
        return lib.pnp_variable_density_masks(accel, st, seeds, ah, aw, power, out, B, H, W, None)

    for kw in ({"accel": None}, {"seeds": None}, {"out": None}, {"B": 0}, {"B": -3}, {"st": -1}, {"H": 1}, {"W": 1025},
               {"H": 2000}, {"ah": -1}, {"aw": -1}, {"ah": 65}, {"aw": 65}, {"power": -1}, {"power": 17},
               {"accel": M + 8}, {"accel": M - 2}, {"seeds": M + 2 * 64 * 64 - 8}, {"seeds": M - 8}, {"out": S + 8},
               {"out": A - 100}):
        assert masks(**kw) < 0, kw
        assert b"pnp_variable_density_masks" in lib.pnp_last_error(), kw


def test_call_before_init_fails_with_a_message():
    lib = _lib.load()
    if _lib._inited:
        pytest.skip("the library was initialised by an earlier test in this process")
    assert lib.pnp_variable_density_masks(1 << 20, 0, 1 << 24, 0, 0, 3, 1 << 30, 1, 8, 8, None) < 0
    assert b"pnp_init" in lib.pnp_last_error()
