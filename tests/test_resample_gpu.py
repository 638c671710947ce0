"""fmri_image_resample on the GPU: native-resolution uint8 images -> Pillow resize (BILINEAR / BICUBIC) -> shifted /
flipped, normalised fp32 NCHW.
  * against Pillow itself: the output is torch.equal to fmri_image_pipeline applied to PIL.Image.resize's uint8 result
    (after PIL's crop and torchvision's CenterCrop geometry), for uniform and ragged batches of sizes, channel counts
    and crop windows, with and without flip / shift;
  * Hr = Hs, Wr = Ws and no crop: bit-identical to fmri_image_pipeline on the source; two calls: the same bits;
  * ResidentStimuli.batch (with crop windows) and Prefetcher (ragged host batches): the same bits as a direct call;
  * bad descriptors and bands larger than FMRI_RESAMPLE_MAX_SMEM raise FmriError with nothing launched;
  * with FMRI_REFERENCE_ROOT naming a checkout whose data_preprocessing.data_loader imports: against the Stage-I COCO
    transform built from it.
"""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from thesis_fmri_reconstruction_b200 import data
from thesis_fmri_reconstruction_b200 import lib as L
from test_resample_cpu import _WIDE

Image = pytest.importorskip("PIL.Image")
pytestmark = pytest.mark.gpu
MEAN, STD = (0.5, 0.4, 0.3), (0.5, 0.25, 0.2)
PIL_FILTERS = {"bilinear": Image.Resampling.BILINEAR, "bicubic": Image.Resampling.BICUBIC}
EDGE_CROPS = [(0, 0, 200, 300), (280, 340, 200, 300), (0, 150, 480, 200), (130, 0, 200, 640), (479, 0, 1, 640),
              (0, 639, 480, 1)]

# name: (source shapes, crop windows or None, size, resize)
CASES = {
    "480x640_to_64sq": ([(480, 640, 3), (480, 640, 3), (480, 640, 3)], None, (64, 64), None),
    "coco_mix_to_100sq": ([(480, 640, 3), (640, 480, 3), (427, 640, 1), (333, 500, 3)], None, (100, 100), None),
    "375sq_to_64sq": ([(375, 375, 3)] * 2, None, (64, 64), None),
    "50sq_to_64sq_up": ([(50, 50, 3)] * 2, None, (64, 64), None),
    "7x13_to_5x29": ([(7, 13, 3), (7, 13, 3)], None, (5, 29), None),
    "grey_480x640_to_64sq": ([(480, 640, 1)] * 2, None, (64, 64), None),
    "1x1_to_5x3": ([(1, 1, 3), (1, 1, 1)], None, (5, 3), None),
    "1x300_to_7x20": ([(1, 300, 3), (1, 300, 1)], None, (7, 20), None),
    "300x2_to_3x50_vertical_first": ([(300, 2, 3), (300, 2, 1)], None, (3, 50), None),
    "1000x9_to_64x5_vertical_first": ([(1000, 9, 3), (1000, 9, 1)], None, (64, 5), None),
    "2x999_to_1x64": ([(2, 999, 3)], None, (1, 64), None),
    "resize_64_center_crop_64sq": ([(480, 640, 3), (640, 480, 3), (333, 500, 1), (375, 375, 3)], None, (64, 64), 64),
    "resize_72_center_crop_56x48": ([(480, 640, 3), (640, 480, 1), (333, 500, 3)], None, (56, 48), 72),
    "resize_80x72_center_crop_64x48": ([(480, 640, 3), (333, 500, 1)], None, (64, 48), (80, 72)),
    "crops_touching_every_edge": ([(480, 640, 3)] * len(EDGE_CROPS), EDGE_CROPS, (64, 48), None),
    "random_resized_crops_ragged": ([(480, 640, 3), (640, 480, 3), (427, 640, 1), (375, 375, 3), (333, 500, 1)], "rrc",
                                    (64, 64), None),
}


def _images(shapes, seed):
    g = torch.Generator().manual_seed(seed)
    return [torch.randint(0, 256, s, generator=g, dtype=torch.uint8) for s in shapes]


def _aug(n, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.tensor([i % 2 for i in range(n)], dtype=torch.int32), torch.randint(-5, 6, (n, 2), generator=g,
                                                                                     dtype=torch.int32)


def _rrc_crops(imgs, seed):
    from torchvision.transforms import RandomResizedCrop

    torch.manual_seed(seed)
    return [RandomResizedCrop.get_params(t.permute(2, 0, 1), (0.08, 1.0), (3 / 4, 4 / 3)) for t in imgs]


def _pillow(img, crop, size, resize, filter):
    """uint8 [H, W, C] as PIL / torchvision compute it: crop, Resize(resize or size), CenterCrop(size)."""
    a = img.numpy()
    im = Image.fromarray(a if a.shape[2] == 3 else a[:, :, 0])
    if crop is not None:
        t, l, h, w = crop
        im = im.crop((l, t, l + w, t + h))
    Hr, Wr = size if resize is None else data.resized_size(im.height, im.width, resize)
    im = im.resize((Wr, Hr), PIL_FILTERS[filter])
    oy, ox, H, W = data.center_crop(Hr, Wr, size)
    return torch.from_numpy(np.array(np.asarray(im).reshape(Hr, Wr, -1)[oy:oy + H, ox:ox + W]))


def _expected(imgs, crops, size, resize, filter, flip, shift):
    """fmri_image_pipeline on Pillow's uint8 results, one image at a time (channel counts may differ)."""
    base = data.DevicePipeline(MEAN, STD)
    out = []
    for i, img in enumerate(imgs):
        u8 = _pillow(img, None if crops is None else crops[i], size, resize, filter)[None].cuda()
        out.append(base(u8, None if flip is None else flip[i:i + 1], None if shift is None else shift[i:i + 1]))
    return torch.cat(out)


@pytest.mark.parametrize("aug", [False, True], ids=["plain", "flip_shift"])
@pytest.mark.parametrize("filter", list(PIL_FILTERS))
@pytest.mark.parametrize("name", list(CASES))
def test_resample_equals_pillow_then_image_pipeline(name, filter, aug):
    shapes, crops, size, resize = CASES[name]
    imgs = _images(shapes, 11)
    if crops == "rrc":
        crops = _rrc_crops(imgs, 12)
    flip, shift = _aug(len(imgs), 13) if aug else (None, None)
    pipe = data.DevicePipeline(MEAN, STD, size=size, resample=filter, resize=resize)
    got = pipe([t.cuda() for t in imgs], flip, shift, crops=crops)
    want = _expected(imgs, crops, size, resize, filter, flip, shift)
    assert got.shape == want.shape
    assert torch.equal(got, want), (got - want).abs().max().item()


@pytest.mark.parametrize("filter", list(PIL_FILTERS))
def test_equal_size_is_bit_identical_to_image_pipeline(filter):
    for C in (3, 1):
        u8 = torch.stack(_images([(64, 48, C)] * 5, 20 + C)).cuda()
        flip, shift = _aug(5, 21)
        for f, s in ((None, None), (flip, shift)):
            a = data.DevicePipeline(MEAN, STD)(u8, f, s)
            b = data.DevicePipeline(MEAN, STD, size=(64, 48), resample=filter)(u8, f, s)
            assert torch.equal(a, b), C


def test_two_calls_give_the_same_bits():
    shapes, _, size, resize = CASES["resize_64_center_crop_64sq"]
    imgs = [t.cuda() for t in _images(shapes, 30)]
    flip, shift = _aug(len(imgs), 31)
    for filter in PIL_FILTERS:
        pipe = data.DevicePipeline(MEAN, STD, size=size, resample=filter, resize=resize)
        assert torch.equal(pipe(imgs, flip, shift), pipe(imgs, flip, shift))


def _pair(seed, **kw):
    mk = lambda: data.DevicePipeline(MEAN, STD, random_flip=True, max_shift=4, generator=torch.Generator().manual_seed(seed),
                                     size=(64, 64), **kw)
    return mk(), mk()


def test_resident_stimuli_batch_equals_direct_call():
    imgs = [t.numpy() for t in _images([(480, 640, 3), (640, 480, 3), (333, 500, 1), (375, 375, 3), (64, 64, 3)], 40)]
    imgs.append(imgs[2][:, :, 0])                                        # a grey image given as [H, W]
    stim = data.ResidentStimuli(imgs)
    direct = lambda idx: [torch.from_numpy(np.ascontiguousarray(imgs[i].reshape(imgs[i].shape[0], imgs[i].shape[1], -1)))
                          for i in idx]
    for kw in (dict(resample="bilinear"), dict(resample="bicubic", resize=72)):
        pa, pb = _pair(41, **kw)
        for idx in ([3, 0, 2, 2, 5], [1], [4, 3, 2, 1, 0, 5]):
            x = stim.batch(idx, pa)
            flip, shift = pb.draw(len(idx))
            assert torch.equal(x, pb([t.cuda() for t in direct(idx)], flip, shift)), (kw, idx)
    # RandomResizedCrop draws passed straight in
    pa, pb = _pair(42, resample="bilinear")
    idx = [0, 1, 2, 3, 5, 0]
    crops = _rrc_crops(direct(idx), 43)
    x = stim.batch(idx, pa, crops=crops)
    flip, shift = pb.draw(len(idx))
    assert torch.equal(x, pb([t.cuda() for t in direct(idx)], flip, shift, crops=crops))
    assert torch.equal(x, _expected(direct(idx), crops, (64, 64), None, "bilinear", flip, shift))


def test_prefetcher_ragged_host_batches_equal_direct_call():
    shapes = [[(480, 640, 3), (50, 50, 1), (640, 480, 3)], [(64, 64, 3), (427, 640, 1)], [(100, 80, 3)] * 3]
    host = [[t.numpy() for t in _images(s, 50 + i)] for i, s in enumerate(shapes)]
    batches = [(b, {"fmri": torch.full((len(b), 7), float(i))}) for i, b in enumerate(host)]
    pa, pb = _pair(51, resample="bicubic")
    seen = 0
    for i, (x, ex) in enumerate(data.Prefetcher(batches, pa)):
        flip, shift = pb.draw(len(host[i]))
        assert torch.equal(x, pb([torch.from_numpy(a).cuda() for a in host[i]], flip, shift)), i
        assert ex["fmri"].is_cuda and float(ex["fmri"][0, 0]) == float(i)
        seen += 1
    assert seen == 3


def test_band_at_the_shared_memory_limit_runs():
    """The widest one-row window FMRI_RESAMPLE_MAX_SMEM allows (1 x (_WIDE - 1) grey -> 1 x 64 BICUBIC) runs and
    matches Pillow; one pixel wider is refused (see test_argument_errors_raise_and_launch_nothing)."""
    img = _images([(1, _WIDE - 1, 1)], 60)
    got = data.DevicePipeline(MEAN, STD, size=(1, 64), resample="bicubic")([img[0].cuda()])
    assert torch.equal(got, _expected(img, None, (1, 64), None, "bicubic", None, None))


def _errs(fn):
    before = L.launch_count()
    with pytest.raises(L.FmriError):
        fn()
    torch.cuda.synchronize()
    assert L.launch_count() == before


def test_argument_errors_raise_and_launch_nothing():
    buf = torch.zeros(480 * 640 * 3, dtype=torch.uint8, device="cuda")
    out = torch.empty(1, 3, 64, 64, device="cuda")
    ws = torch.empty(L.image_resample_workspace(1), dtype=torch.uint8, device="cuda")
    ok = (0, 1920, 480, 640, 3, 64, 64, 0, 0)

    def call(entries, o=out, w=ws, b=buf, filter="bilinear"):
        L.image_resample(b, L.image_window_table(entries), filter, None, None, MEAN, STD, o, w)

    _errs(lambda: call([(0, 1920, 480, 640, 2, 64, 64, 0, 0)]))              # channels
    _errs(lambda: call([(0, 1920, 0, 640, 3, 64, 64, 0, 0)]))                # empty window
    _errs(lambda: call([(1, 1920, 480, 640, 3, 64, 64, 0, 0)]))              # past the end of the buffer
    _errs(lambda: call([(0, 1921, 480, 640, 3, 64, 64, 0, 0)]))              # pitch runs past the end
    _errs(lambda: call([(0, 1919, 480, 640, 3, 64, 64, 0, 0)]))              # pitch < W C
    _errs(lambda: call([(0, 1920, 480, 640, 3, 64, 80, 0, 17)]))             # output leaves the resize
    _errs(lambda: call([ok], filter="lanczos"))
    _errs(lambda: call([ok], w=ws[:8]))                                       # workspace too small
    _errs(lambda: call([ok], w=ws[1:]))                                       # workspace misaligned
    _errs(lambda: call([ok, ok]))                                             # two descriptors, one output image
    _errs(lambda: call([ok], b=buf.cpu()))                                    # host buffer
    _errs(lambda: call([(0, _WIDE, 1, _WIDE, 1, 1, 64, 0, 0)], o=torch.empty(1, 3, 1, 64, device="cuda"),
                       filter="bicubic"))                                     # band larger than FMRI_RESAMPLE_MAX_SMEM
    pipe = data.DevicePipeline(MEAN, STD, size=(64, 64), resample="bilinear")
    _errs(lambda: pipe([buf.view(480, 640, 3)], crops=[(400, 0, 100, 100)]))  # crop window leaves the image
    _errs(lambda: data.DevicePipeline(MEAN, STD, size=(64, 64))([buf.view(480, 640, 3)], crops=[(0, 0, 10, 10)]))
    _errs(lambda: data.DevicePipeline(MEAN, STD)(buf.view(1, 480, 640, 3), crops=[(0, 0, 10, 10)]))
    _errs(lambda: data.DevicePipeline(MEAN, STD, size=(64, 64), resample="bilinear", resize=32)([buf.view(480, 640, 3)]))


_REF = os.environ.get("FMRI_REFERENCE_ROOT")
_LOADER = os.path.join(_REF, "data_preprocessing", "data_loader.py") if _REF else None


def _loader_imports():
    if not (_LOADER and os.path.exists(_LOADER)):
        return False
    r = subprocess.run([sys.executable, "-c", "import sys; sys.path.insert(0, sys.argv[1]); import data_preprocessing.data_loader",
                        _REF], cwd=_REF, capture_output=True)
    return r.returncode == 0


@pytest.mark.skipif(not _loader_imports(),
                    reason="needs FMRI_REFERENCE_ROOT naming a checkout whose data_preprocessing.data_loader imports")
def test_resample_matches_reference_stage1_transform(tmp_path):
    """The Stage-I COCO transform (train_vgan_stage1.py:161-171: torchvision Resize on the PIL image, ToTensor, the
    reference's own GreyToColor, Normalize) run in a child process whose path holds only the reference tree (its
    `configs` package would clash with this repository's). ToTensor divides by 255 where the kernel multiplies by 1/255,
    so the comparison allows one rounding of the [0, 1] value: 1e-6 after normalisation."""
    imgs = [t.numpy() for t in _images([(480, 640, 3), (640, 480, 3), (427, 640, 1)], 70)]
    np.savez(tmp_path / "in.npz", *imgs)
    code = ("import sys, numpy as np, torch; sys.path.insert(0, sys.argv[1]);"
            "from PIL import Image; from torchvision import transforms as T;"
            "from data_preprocessing.data_loader import GreyToColor;"
            "x = np.load(sys.argv[2]); s = int(sys.argv[4]); f = T.InterpolationMode(sys.argv[5]);"
            "t = T.Compose([T.Resize((s, s), f), T.ToTensor(), GreyToColor(), T.Normalize((0.5,) * 3, (0.5,) * 3)]);"
            "np.save(sys.argv[3], np.stack([t(Image.fromarray(a if a.shape[2] == 3 else a[:, :, 0])).numpy() "
            "for a in (x[k] for k in sorted(x.files, key=lambda k: int(k.split('_')[1])))]))")
    for res, filter in ((64, "bilinear"), (100, "bicubic")):
        subprocess.run([sys.executable, "-c", code, _REF, str(tmp_path / "in.npz"), str(tmp_path / "out.npy"), str(res),
                        filter], check=True, cwd=_REF)
        ref = torch.from_numpy(np.load(tmp_path / "out.npy"))
        got = data.DevicePipeline((0.5,) * 3, (0.5,) * 3, size=(res, res), resample=filter)(
            [torch.from_numpy(a).cuda() for a in imgs])
        err = (got.cpu().double() - ref.double()).abs().max().item()
        print(f"resample vs the reference's Stage-I transform at {res} ({filter}): max |error| {err:.3g}")
        assert err < 1e-6, err
