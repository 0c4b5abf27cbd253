"""The float64 measurement reference (tests/measure_reference.py) on its own, and the simulator's C-ABI without a GPU."""
import numpy as np
import pytest

from dt4image_restoration_b200 import _lib, synth
from measure_reference import acs_cols, cartesian_mask, noise, philox4x32_10, simulate


def _words(c):
    return [int(np.asarray(w).reshape(-1)[0]) for w in c]


@pytest.mark.parametrize("counter,key,expect", [
    ((0, 0, 0, 0), (0, 0), (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
    ((0xFFFFFFFF,) * 4, (0xFFFFFFFF, 0xFFFFFFFF), (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)),
    ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0),
     (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1)),
])
def test_philox_known_answers(counter, key, expect):
    assert _words(philox4x32_10(counter, key)) == list(expect)


def test_philox_is_vectorised_elementwise():
    ctr = np.array([0, 5, 0xFFFFFFFF], dtype=np.uint64)
    vec = philox4x32_10((ctr, 1, 0, 0), (3, 9))
    for n, c in enumerate(ctr):
        assert _words(philox4x32_10((int(c), 1, 0, 0), (3, 9))) == [int(w[n]) for w in vec]


def test_noise_statistics():
    n_r, n_i = noise(12345, 1000, 1000)               # 10^6 samples of each
    for n in (n_r, n_i):
        assert abs(n.mean()) < 5e-3 and abs(n.var() - 1.0) < 1e-2
    assert abs(np.corrcoef(n_r.ravel(), n_i.ravel())[0, 1]) < 5e-3
    assert abs(np.corrcoef(n_r[:, :-1].ravel(), n_r[:, 1:].ravel())[0, 1]) < 5e-3   # neighbouring samples


def test_noise_depends_on_seed_and_both_seed_words():
    a = noise(1, 8, 8)[0]
    assert not np.array_equal(a, noise(2, 8, 8)[0])
    assert not np.array_equal(a, noise(1 + (1 << 32), 8, 8)[0])
    assert np.array_equal(noise(-1, 4, 4)[0], noise((1 << 64) - 1, 4, 4)[0])


@pytest.mark.parametrize("H,W", [(32, 32), (45, 51), (64, 128), (2, 3)])
def test_noise_off_equals_synth_make_item(H, W):
    gt = synth.phantom(H, W, 3)
    for mask in (synth.radial_mask(H, W, 0.3), synth.cartesian_mask(H, W, 4, 3)):
        item = synth.make_item(gt, mask, 0.0, 3)
        k = synth.centered_fft2(gt.astype(np.float64))
        y0, aty0, x0 = simulate(gt, mask, 0.0, 99)
        y0_s = k * mask.astype(np.float64)
        assert np.abs(y0 - y0_s).max() <= 1e-12
        assert np.abs(aty0 - synth.centered_ifft2(y0_s)).max() <= 1e-12
        ri = lambda z: np.stack([z.real, z.imag], axis=-1).astype(np.float32).reshape(1, 1, H, W, 2)
        assert np.array_equal(ri(y0), item["y0"]) and np.array_equal(ri(aty0), item["ATy0"])
        assert np.array_equal(ri(x0), item["x0"])


def test_noise_is_added_only_under_the_mask():
    gt = synth.phantom(16, 16, 0)
    mask = synth.cartesian_mask(16, 16, 2, 0)
    y_off = simulate(gt, mask, 0.0, 5)[0]
    y_on = simulate(gt, mask, 10.0, 5)[0]
    n_r, n_i = noise(5, 16, 16)
    assert np.all(y_on[mask == 0] == 0)
    assert np.abs((y_on - y_off)[mask != 0] - (10 / 255) * (n_r + 1j * n_i)[mask != 0]).max() <= 1e-14


@pytest.mark.parametrize("H,W,accel", [(256, 256, 4), (45, 51, 2), (2, 3, 8), (1000, 37, 3), (16, 1024, 8), (64, 64, 1)])
def test_cartesian_mask_invariants(H, W, accel):
    a = acs_cols(W)
    m = cartesian_mask(H, W, accel, 7, a)
    assert m.dtype == np.uint8 and m.shape == (H, W)
    assert np.all(m == m[0:1])                                    # depends on the column only
    n_keep = max(1, W // accel)
    assert int(m[0].sum()) == n_keep
    n_acs = min(n_keep, a)
    c0 = W // 2 - n_acs // 2
    assert np.all(m[0, c0:c0 + n_acs] == 1)                         # ACS band
    assert np.array_equal(m, cartesian_mask(H, W, accel, 7, a))
    if n_keep - n_acs > 0 and W - n_acs > n_keep - n_acs:
        assert not all(np.array_equal(m, cartesian_mask(H, W, accel, s, a)) for s in (8, 9, 10))


def test_cartesian_mask_same_structure_as_synth():
    for (H, W, accel) in ((64, 64, 4), (128, 96, 8)):
        ref = synth.cartesian_mask(H, W, accel, 0)
        got = cartesian_mask(H, W, accel, 0, acs_cols(W))
        assert ref[0].sum() == got[0].sum()
        n_acs = min(max(1, W // accel), acs_cols(W))
        c0 = W // 2 - n_acs // 2
        assert np.all(ref[0, c0:c0 + n_acs] == got[0, c0:c0 + n_acs])


def test_per_image_accel():
    ms = [cartesian_mask(32, 64, a, 3, acs_cols(64)) for a in (1, 2, 4, 8)]
    assert [int(m[0].sum()) for m in ms] == [64, 32, 16, 8]


def test_c_abi_rejects_bad_arguments_without_a_gpu():
    """Argument checks run before the init check, so they answer on a machine without a GPU (fake addresses are never
    dereferenced: every call below is refused)."""
    lib = _lib.load()
    A, M, S, K = 1 << 20, 1 << 24, 1 << 26, 1 << 27                  # gt, mask, sigma, seeds
    Y, X, T = 1 << 30, 1 << 31, 1 << 32                              # y0, x0, aty0 (64x64 c64 images: 32 KiB each)

    def sim(gt=A, mask=M, sig=S, seeds=K, y0=Y, x0=X, at=T, B=2, H=64, W=64, gs=4096, ms=4096, ss=1):
        return lib.pnp_simulate_measurements(gt, gs, mask, ms, sig, ss, seeds, y0, x0, at, B, H, W, None)

    for kw in ({"gt": None}, {"mask": None}, {"sig": None}, {"seeds": None}, {"y0": None}, {"x0": None}, {"B": 0},
               {"B": -1}, {"H": 1}, {"W": 1025}, {"H": 2000}, {"gs": -1}, {"ss": -1}, {"y0": A + 4096},
               {"x0": M + 100}, {"at": Y + 8}, {"x0": Y}, {"y0": X - 8}):
        rc = sim(**kw)
        assert rc < 0, kw
        assert b"pnp_simulate_measurements" in lib.pnp_last_error(), kw

    def masks(accel=A, seeds=K, out=Y, acs=5, B=2, H=64, W=64, st=1):
        return lib.pnp_cartesian_masks(accel, st, seeds, acs, out, B, H, W, None)

    for kw in ({"accel": None}, {"seeds": None}, {"out": None}, {"acs": 0}, {"B": 0}, {"H": 1}, {"W": 1025}, {"st": -1}):
        assert masks(**kw) < 0, kw
        assert b"pnp_cartesian_masks" in lib.pnp_last_error(), kw


def test_calls_before_init_fail_with_a_message():
    lib = _lib.load()
    if _lib._inited:
        pytest.skip("the library was initialised by an earlier test in this process")
    assert lib.pnp_simulate_measurements(1 << 20, 0, 1 << 24, 0, 1 << 26, 0, 1 << 27, 1 << 30, 1 << 31, None, 1, 8, 8,
                                         None) < 0
    assert b"pnp_init" in lib.pnp_last_error()
    assert lib.pnp_cartesian_masks(1 << 20, 0, 1 << 27, 1, 1 << 30, 1, 8, 8, None) < 0
    assert b"pnp_init" in lib.pnp_last_error()
