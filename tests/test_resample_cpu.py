"""CPU checks of the PIL-compatible resample: the numpy restatement of Pillow's 8-bit resampler
(tests/pil_resample_reference.py) against PIL.Image.resize byte for byte, torchvision's Resize / CenterCrop /
RandomResizedCrop on PIL images against the restatement driven by data.resample_windows, and the C ABI of
fmri_image_resample (exports, workspace query, every argument error refused before anything touches the device)."""
import ctypes
import math

import numpy as np
import pytest
import torch

import pil_resample_reference as R
from thesis_fmri_reconstruction_b200 import data
from thesis_fmri_reconstruction_b200 import lib as L

Image = pytest.importorskip("PIL.Image")
PIL_FILTERS = {"bilinear": Image.Resampling.BILINEAR, "bicubic": Image.Resampling.BICUBIC}
FILTERS = list(PIL_FILTERS)


def _img(shape, seed):
    return np.random.default_rng(seed).integers(0, 256, shape, dtype=np.uint8)


def _pil(a, out_hw, filter, box=None):
    return np.asarray(Image.fromarray(a).resize((out_hw[1], out_hw[0]), PIL_FILTERS[filter], box=box))


# (source shape, output (H, W), box or None): downscale, upscale, non-integer and mixed scales, 1-pixel and very elongated
# images, fractional boxes and boxes touching every edge of the source
RESIZE_CASES = {
    "480x640_to_64sq": ((480, 640), (64, 64), None),
    "333x500_to_100sq": ((333, 500), (100, 100), None),
    "375sq_to_64sq": ((375, 375), (64, 64), None),
    "50sq_to_64sq_up": ((50, 50), (64, 64), None),
    "7x13_to_5x29": ((7, 13), (5, 29), None),
    "64sq_identity": ((64, 64), (64, 64), None),
    "1x1_to_5x3": ((1, 1), (5, 3), None),
    "1x300_to_7x20": ((1, 300), (7, 20), None),
    "300x2_to_3x50": ((300, 2), (3, 50), None),
    "2x999_to_1x64": ((2, 999), (1, 64), None),
    "tall_1000x9_to_64x5": ((1000, 9), (64, 5), None),                  # Image.resize takes the vertical pass first
    "box_fractional": ((480, 640), (64, 64), (13.25, 7.5, 619.0, 477.75)),
    "box_fractional_up": ((50, 50), (64, 64), (0.5, 1.0, 49.75, 49.0)),
    "box_top_left": ((333, 500), (100, 100), (0, 0, 250, 160)),
    "box_bottom_right": ((333, 500), (100, 100), (250, 173, 500, 333)),
    "box_full_height": ((333, 500), (64, 48), (100, 0, 300, 333)),
    "box_full_width": ((333, 500), (48, 64), (0, 100, 500, 300)),
}


@pytest.mark.parametrize("filter", FILTERS)
@pytest.mark.parametrize("channels", [3, 1], ids=["rgb", "l"])
@pytest.mark.parametrize("name", list(RESIZE_CASES))
def test_restatement_matches_pillow(name, channels, filter):
    shape, out, box = RESIZE_CASES[name]
    a = _img(shape + ((3,) if channels == 3 else ()), sum(map(ord, name)))
    want = _pil(a, out, filter, box)
    got = R.resize(a, out, filter, box)
    assert got.shape == want.shape and np.array_equal(got, want), np.abs(got.astype(int) - want).max()


@pytest.mark.parametrize("filter", FILTERS)
@pytest.mark.parametrize("window", [(0, 0, 200, 300), (280, 340, 200, 300), (0, 150, 480, 200), (130, 0, 200, 640),
                                    (479, 0, 1, 640), (0, 639, 480, 1)],
                         ids=["top_left", "bottom_right", "full_height", "full_width", "last_row", "last_column"])
def test_crop_then_resize_clamps_at_the_crop(window, filter):
    """PIL's crop-then-resize filters the crop alone: its taps stop at the crop's edges, not the image's."""
    a = _img((480, 640, 3), 3)
    t, l, h, w = window
    want = np.asarray(Image.fromarray(a).crop((l, t, l + w, t + h)).resize((48, 64), PIL_FILTERS[filter]))
    assert np.array_equal(R.resize(a[t:t + h, l:l + w], (64, 48), filter), want)


# ------------------------------------------------------------------------------------------------ torchvision geometry
def test_resized_size_matches_torchvision():
    from torchvision.transforms.functional import _compute_resized_output_size as tv

    for h, w in ((480, 640), (640, 480), (333, 500), (375, 375), (1, 7), (7, 1), (427, 640), (612, 612)):
        for size in (64, 100, 224, 256, 333, [80], (64, 48), [100, 100]):
            want = tv((h, w), list(size) if not isinstance(size, int) else [size])
            assert list(data.resized_size(h, w, size)) == want, (h, w, size)


def _tv_case(name, filter, a):
    """(torchvision output uint8 HWC, size, resize, crops) for one transform chain on one PIL image."""
    from torchvision import transforms as T

    im = Image.fromarray(a if a.shape[2] == 3 else a[:, :, 0])
    mode = {"bilinear": T.InterpolationMode.BILINEAR, "bicubic": T.InterpolationMode.BICUBIC}[filter]
    h, w = a.shape[:2]
    if name == "resize_pair":
        return T.Resize((64, 80), mode)(im), (64, 80), None, None
    if name == "resize_short_side_center_crop":
        return T.CenterCrop(64)(T.Resize(64, mode)(im)), (64, 64), 64, None
    if name == "resize_short_side_center_crop_rect":
        return T.CenterCrop((56, 48))(T.Resize(72, mode)(im)), (56, 48), 72, None
    if name == "resize_pair_center_crop":
        return T.CenterCrop((64, 48))(T.Resize((80, 72), mode)(im)), (64, 48), (80, 72), None
    if name == "center_crop_then_resize":
        return T.Resize((64, 64), mode)(T.CenterCrop(300)(im)), (64, 64), None, [data.center_crop(h, w, 300)]
    if name == "random_resized_crop":
        rrc = T.RandomResizedCrop(64, interpolation=mode)
        torch.manual_seed(h * w + a.shape[2])
        p = rrc.get_params(im, rrc.scale, rrc.ratio)
        return T.functional.resized_crop(im, *p, [64, 64], mode), (64, 64), None, [p]
    raise KeyError(name)


@pytest.mark.parametrize("filter", FILTERS)
@pytest.mark.parametrize("name", ["resize_pair", "resize_short_side_center_crop", "resize_short_side_center_crop_rect",
                                  "resize_pair_center_crop", "center_crop_then_resize", "random_resized_crop"])
def test_torchvision_geometry_matches_restatement(name, filter):
    pytest.importorskip("torchvision")
    for shape in ((480, 640, 3), (640, 480, 3), (333, 500, 1), (375, 375, 3)):
        a = _img(shape, shape[0] + shape[2])
        want, size, resize, crops = _tv_case(name, filter, a)
        want = np.asarray(want).reshape(size[0], size[1], -1)
        buf, entries = data.pack_images([torch.from_numpy(a)])
        (win,) = data.resample_windows(entries, size, resize, crops)
        got = R.resample_window(buf.numpy(), win, size, filter)
        assert got.shape == want.shape and np.array_equal(got, want), (shape, win)


def test_resample_windows_geometry():
    entries = [(0, 480, 640, 3), (921600, 333, 500, 1)]
    # Resize(64) then CenterCrop(64): the shorter side becomes 64, the output is the centre of the longer one
    assert data.resample_windows(entries, (64, 64), 64) == [(0, 1920, 480, 640, 3, 64, 85, 0, 10),
                                                            (921600, 500, 333, 500, 1, 64, 96, 0, 16)]
    # a crop window becomes an offset into the image with the image's pitch
    assert data.resample_windows(entries[:1], (32, 32), None, [(10, 20, 100, 200)]) == [
        ((10 * 640 + 20) * 3, 1920, 100, 200, 3, 32, 32, 0, 0)]
    assert data.center_crop(480, 640, 300) == (90, 170, 300, 300)
    assert data.center_crop(5, 5, (2, 2)) == (2, 2, 2, 2)                 # round(1.5) = 2, as torchvision
    with pytest.raises(L.FmriError):
        data.center_crop(64, 85, 100)                                     # torchvision would pad
    with pytest.raises(L.FmriError):
        data.resample_windows(entries[:1], (32, 32), None, [(400, 0, 100, 100)])
    with pytest.raises(L.FmriError):
        data.resample_windows(entries[:1], (32, 32), None, [(0, 0, 0, 100)])
    with pytest.raises(L.FmriError):
        data.resample_windows(entries, (32, 32), None, [(0, 0, 10, 10)])
    with pytest.raises(L.FmriError):
        data.resample_windows(entries[:1], (64, 64), 32)                  # Resize(32) is smaller than the 64 x 64 crop


def test_pipeline_options_refused():
    with pytest.raises(L.FmriError):
        data.DevicePipeline(size=(64, 64), resample="lanczos")
    with pytest.raises(L.FmriError):
        data.DevicePipeline(resample="bilinear")                           # needs size
    with pytest.raises(L.FmriError):
        data.DevicePipeline(size=(64, 64), resize=64)                     # resize= belongs to the PIL resample
    p = data.DevicePipeline(size=(64, 64))
    assert p.resample is None and p.resize is None                        # the default stays the skimage Rescale


# ------------------------------------------------------------------------------------------------ C ABI
def test_band_bytes_example():
    assert band_bytes(480, 640, 3, 64, 64, 64, 64, "bicubic") == 17296                # the example in the header


def test_resample_exports_and_workspace_query():
    names = L.header_functions()
    assert "fmri_image_resample" in names and "fmri_image_resample_workspace" in names
    c = ctypes.CDLL(L.LIB_PATH)
    assert hasattr(c, "fmri_image_resample") and hasattr(c, "fmri_image_resample_workspace")
    assert ctypes.sizeof(L.ImageWindow) == 48
    assert L.image_resample_workspace(0) == 0 and L.image_resample_workspace(-3) == 0
    assert L.image_resample_workspace(256) == 256 * 48
    assert L.RESAMPLE_FILTERS == {"bilinear": int(Image.Resampling.BILINEAR), "bicubic": int(Image.Resampling.BICUBIC)}


def _max_smem():
    import re

    return int(re.search(r"#define\s+FMRI_RESAMPLE_MAX_SMEM\s+(\d+)", open(L.HEADER_PATH).read()).group(1))


def band_bytes(h, w, c, Hr, Wr, H, W, filter, ty=1):
    """Shared memory of a band of ty output rows, as include/fmri_b200.h states it."""
    a16 = lambda b: (b + 15) // 16 * 16
    s = {"bilinear": 1, "bicubic": 2}[filter]
    sup_x, sup_y = s * max(w / Wr, 1.0), s * max(h / Hr, 1.0)
    kx, ky = 2 * math.ceil(sup_x) + 1, 2 * math.ceil(sup_y) + 1
    first = ty * w if h > 100 * w and Hr < h else min(h, int((ty - 1) * (h / Hr) + 2 * sup_y) + 2) * W
    return a16(4 * W * kx) + a16(8 * W) + a16(4 * ty * ky) + a16(8 * ty) + first * c


def _call(entries, N=None, H=64, W=64, filter=2, src_bytes=480 * 640 * 3, ws_bytes=None, ws=64, src=16, dst=16):
    table = L.image_window_table(entries)
    N = len(entries) if N is None else N
    ws_bytes = L.image_resample_workspace(max(N, 1)) if ws_bytes is None else ws_bytes
    return L.load().fmri_image_resample(ctypes.c_void_p(src), ctypes.c_size_t(src_bytes), table, N, H, W, filter, None,
                                        None, None, None, ctypes.c_void_p(dst), ctypes.c_void_p(ws),
                                        ctypes.c_size_t(ws_bytes), None)


OK = (0, 1920, 480, 640, 3, 64, 64, 0, 0)
# the widest one-row grey window the shared memory allows when resized to 1 x 64 with BICUBIC, and one pixel wider
_WIDE = next(w for w in range(4096, 32769) if band_bytes(1, w, 1, 1, 64, 1, 64, "bicubic") > _max_smem())


@pytest.mark.parametrize("case, want", [
    (dict(entries=[OK], N=0), "ARG"),
    (dict(entries=[OK], H=0), "ARG"),
    (dict(entries=[OK], W=40000), "ARG"),
    (dict(entries=[OK], src=0), "ARG"),
    (dict(entries=[OK], dst=0), "ARG"),
    (dict(entries=[OK], filter=0), "ARG"),                                        # NEAREST
    (dict(entries=[OK], filter=1), "ARG"),                                        # LANCZOS
    (dict(entries=[OK], filter=4), "ARG"),                                        # BOX
    (dict(entries=[(0, 1920, 480, 640, 2, 64, 64, 0, 0)]), "ARG"),                # channels
    (dict(entries=[(0, 1920, 0, 640, 3, 64, 64, 0, 0)]), "ARG"),                  # empty window
    (dict(entries=[(0, 1920, 480, -1, 3, 64, 64, 0, 0)]), "ARG"),
    (dict(entries=[(0, 1920, 480, 640, 3, 0, 64, 0, 0)]), "ARG"),                 # empty resize
    (dict(entries=[(0, 1920, 480, 640, 3, 64, 40000, 0, 0)]), "ARG"),
    (dict(entries=[(0, 1920, 480, 640, 3, 64, 64, -1, 0)]), "ARG"),               # output offset outside the resize
    (dict(entries=[(0, 1920, 480, 640, 3, 64, 64, 0, -1)]), "ARG"),
    (dict(entries=[(0, 1920, 480, 640, 3, 64, 85, 1, 0)]), "ARG"),                # oy + H > Hr
    (dict(entries=[(0, 1920, 480, 640, 3, 64, 85, 0, 22)]), "ARG"),               # ox + W > Wr
    (dict(entries=[(0, 1919, 480, 640, 3, 64, 64, 0, 0)]), "ARG"),                # pitch < W C
    (dict(entries=[(-1, 1920, 480, 640, 3, 64, 64, 0, 0)]), "ARG"),               # negative offset
    (dict(entries=[(1, 1920, 480, 640, 3, 64, 64, 0, 0)]), "ARG"),                # one byte past the buffer
    (dict(entries=[(0, 1921, 480, 640, 3, 64, 64, 0, 0)]), "ARG"),                # pitch runs past the buffer
    (dict(entries=[(0, 1 << 62, 3, 640, 3, 64, 64, 0, 0)]), "ARG"),               # (H - 1) pitch overflows 64 bits
    (dict(entries=[(1 << 40, 1, 1, 1, 1, 64, 64, 0, 0)]), "ARG"),
    (dict(entries=[OK, (0, 1920, 480, 641, 3, 64, 64, 0, 0)]), "ARG"),            # the second window does not fit
    (dict(entries=[OK], ws=0), "WORKSPACE"),
    (dict(entries=[OK], ws_bytes=47), "WORKSPACE"),
    (dict(entries=[OK], ws=68), "ARG"),                                           # not 8-byte aligned
    (dict(entries=[(0, _WIDE, 1, _WIDE, 1, 1, 64, 0, 0)], H=1, filter=3), "UNSUPPORTED"),
    (dict(entries=[OK, (0, 32768, 1, 32768, 1, 1, 64, 0, 0)], H=1), "UNSUPPORTED"),
])
def test_resample_argument_errors_launch_nothing(case, want):
    """Every argument, and the shared-memory limit, is checked on the host before the first CUDA call: no GPU is needed
    to see them refused."""
    before = L.launch_count()
    rc = _call(**case)
    assert rc == {"ARG": -1, "UNSUPPORTED": -2, "WORKSPACE": -4}[want], (rc, L.load().fmri_last_error())
    assert L.launch_count() == before
