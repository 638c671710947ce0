"""CPU checks of the stimulus rescale: the fp64 restatement of skimage.transform.resize (tests/rescale_reference.py) against
a hand-computed case and the properties the resize must have, against real scikit-image when it is importable, and the
C ABI of fmri_image_rescale (exports, workspace query, every argument error refused before anything touches the device)."""
import ctypes

import numpy as np
import pytest

import rescale_reference as R
from thesis_fmri_reconstruction_b200 import lib as L

RNG = np.random.default_rng(5)


def test_resize_hand_computed_8_to_3():
    """One row of 8 pixels -> 3: f = 8/3, sigma = 5/6, radius int(4 sigma + 0.5) = 3, taps exp(-0.72 j^2) normalised,
    mirror boundary; the bilinear taps sit at u = (o + 0.5) 8/3 - 0.5 = 5/6, 7/2, 37/6."""
    s = np.array([0, 10, 40, 90, 160, 250, 30, 70], dtype=np.float64) / 255
    g = np.exp(-0.72 * np.arange(-3, 4) ** 2)
    g /= g.sum()
    taps = {0: [3, 2, 1, 0, 1, 2, 3], 1: [2, 1, 0, 1, 2, 3, 4], 3: [0, 1, 2, 3, 4, 5, 6], 4: [1, 2, 3, 4, 5, 6, 7],
            6: [3, 4, 5, 6, 7, 6, 5], 7: [4, 5, 6, 7, 6, 5, 4]}           # k + j, j = -3..3, mirrored into [0, 7]
    F = {k: float(np.dot(g, s[idx])) for k, idx in taps.items()}
    want = [F[0] / 6 + F[1] * 5 / 6, (F[3] + F[4]) / 2, F[6] * 5 / 6 + F[7] / 6]
    got = R.resize((s * 255).astype(np.uint8)[None, :], (1, 3))
    assert got.shape == (1, 3)
    np.testing.assert_allclose(got[0], want, rtol=0, atol=1e-15)


def test_resize_constant_stays_constant():
    for shape, out in (((37, 23, 3), (10, 9)), ((20, 20, 1), (64, 48)), ((375, 375, 3), (64, 64))):
        img = np.full(shape, 77, dtype=np.uint8)
        np.testing.assert_allclose(R.resize(img, out), 77 / 255, rtol=0, atol=1e-15)


def test_resize_equal_size_is_identity():
    for shape in ((64, 64, 3), (31, 17, 1), (5, 9)):
        img = RNG.integers(0, 256, shape, dtype=np.uint8)
        assert np.array_equal(R.resize(img, shape[:2]), img / 255.0)


def test_resize_mirror_symmetry():
    """Flipping the source flips the result (the taps and the sample grid are symmetric about the image centre)."""
    for shape, out in (((375, 375, 3), (64, 64)), ((50, 41, 1), (64, 13)), ((33, 70, 3), (10, 100))):
        img = RNG.integers(0, 256, shape, dtype=np.uint8)
        r = R.resize(img, out)
        np.testing.assert_allclose(R.resize(img[:, ::-1], out), r[:, ::-1], rtol=0, atol=1e-12)
        np.testing.assert_allclose(R.resize(img[::-1], out), r[::-1], rtol=0, atol=1e-12)


def test_transform_grey_shift_flip_normalise():
    img = RNG.integers(0, 256, (40, 30), dtype=np.uint8)
    base = R.transform([img], (16, 12))[0]
    assert np.array_equal(base[0], base[1]) and np.array_equal(base[0], base[2])       # GreyToColor
    got = R.transform([img[:, :, None]], (16, 12), flip=[1], shift_yx=[(2, -3)], mean=(0.5, 0.4, 0.3), std=(0.5, 0.25, 0.2))[0]
    ys = np.clip(np.arange(16) - 2, 0, 15)
    xs = np.clip(np.arange(12)[::-1] + 3, 0, 11)
    want = (base.numpy()[:, ys][:, :, xs] - np.array([0.5, 0.4, 0.3])[:, None, None]) / np.array([0.5, 0.25, 0.2])[:, None, None]
    np.testing.assert_allclose(got.numpy(), want, rtol=0, atol=1e-15)


def test_restatement_matches_skimage():
    skimage = pytest.importorskip("skimage")
    if "script_harness" in (getattr(skimage, "__file__", "") or ""):
        pytest.skip("only the harness's stand-in for scikit-image is importable")
    from skimage.transform import resize

    for shape, out in (((375, 375, 3), (100, 100)), ((375, 375, 3), (64, 64)), ((500, 333, 3), (64, 64)),
                       ((50, 50, 3), (64, 64)), ((60, 45), (64, 20))):
        img = RNG.integers(0, 256, shape, dtype=np.uint8)
        np.testing.assert_allclose(R.resize(img, out), resize(img, out), rtol=0, atol=1e-12)


# ------------------------------------------------------------------------------------------------ C ABI
def test_rescale_exports_and_workspace_query():
    names = L.header_functions()
    assert "fmri_image_rescale" in names and "fmri_image_rescale_workspace" in names
    c = ctypes.CDLL(L.LIB_PATH)
    assert hasattr(c, "fmri_image_rescale") and hasattr(c, "fmri_image_rescale_workspace")
    assert ctypes.sizeof(L.ImageSrc) == 24
    assert L.image_rescale_workspace(0) == 0 and L.image_rescale_workspace(-3) == 0
    assert L.image_rescale_workspace(256) == 256 * 24


def _call(entries, N=None, H=64, W=64, src_bytes=375 * 375 * 3, ws_bytes=None, ws=64, src=16, dst=16):
    table = L.image_src_table(entries)
    N = len(entries) if N is None else N
    ws_bytes = L.image_rescale_workspace(max(N, 1)) if ws_bytes is None else ws_bytes
    lib = L.load()
    return lib.fmri_image_rescale(ctypes.c_void_p(src), ctypes.c_size_t(src_bytes), table, N, H, W, None, None, None, None,
                                  ctypes.c_void_p(dst), ctypes.c_void_p(ws), ctypes.c_size_t(ws_bytes), None)


@pytest.mark.parametrize("case, want", [
    (dict(entries=[(0, 375, 375, 3)], N=0), "ARG"),
    (dict(entries=[(0, 375, 375, 3)], H=0), "ARG"),
    (dict(entries=[(0, 375, 375, 3)], W=40000), "ARG"),
    (dict(entries=[(0, 375, 375, 3)], src=0), "ARG"),
    (dict(entries=[(0, 375, 375, 3)], dst=0), "ARG"),
    (dict(entries=[(0, 375, 375, 2)]), "ARG"),
    (dict(entries=[(0, 0, 375, 3)]), "ARG"),
    (dict(entries=[(0, 375, -1, 1)]), "ARG"),
    (dict(entries=[(-1, 375, 375, 3)]), "ARG"),
    (dict(entries=[(1, 375, 375, 3)]), "ARG"),                                   # one byte past the buffer
    (dict(entries=[(0, 375, 375, 3), (0, 376, 375, 3)]), "ARG"),                 # the second image does not fit
    (dict(entries=[(1 << 40, 1, 1, 1)]), "ARG"),
    (dict(entries=[(0, 375, 375, 3)], ws=0), "WORKSPACE"),
    (dict(entries=[(0, 375, 375, 3)], ws_bytes=23), "WORKSPACE"),
    (dict(entries=[(0, 375, 375, 3)], ws=68), "ARG"),                            # not 8-byte aligned
])
def test_rescale_argument_errors_launch_nothing(case, want):
    """Every argument is checked on the host before the first CUDA call: no GPU is needed to see them refused."""
    before = L.launch_count()
    rc = _call(**case)
    assert rc == {"ARG": -1, "WORKSPACE": -4}[want], (rc, L.load().fmri_last_error())
    assert L.launch_count() == before
