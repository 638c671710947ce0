"""fmri_image_rescale on the GPU: native-resolution uint8 stimuli -> resized, shifted / flipped, normalised fp32 NCHW.
  * against the fp64 restatement of skimage.transform.resize (tests/rescale_reference.py): 2e-6 absolute on the [0, 1]
    scale (the normalised difference times std); fp32 taps and sums over up to ~30 x 30 source pixels per output pixel;
  * equal sizes: bit-identical to fmri_image_pipeline; two calls: the same bits;
  * ResidentStimuli.batch and Prefetcher (ragged host batches): the same bits as a direct DevicePipeline call;
  * every argument error raises FmriError with nothing launched;
  * with FMRI_REFERENCE_ROOT naming a checkout and real scikit-image importable: against the reference's own Rescale.
"""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import rescale_reference as R
from thesis_fmri_reconstruction_b200 import data
from thesis_fmri_reconstruction_b200 import lib as L

pytestmark = pytest.mark.gpu
MEAN, STD = (0.5, 0.4, 0.3), (0.5, 0.25, 0.2)
TOL = 2e-6

CASES = {
    "375sq_to_100sq": ([(375, 375, 3)] * 4, (100, 100)),
    "375sq_to_64sq": ([(375, 375, 3)] * 4, (64, 64)),
    "500x333_to_64sq": ([(500, 333, 3)] * 3, (64, 64)),
    "50sq_to_64sq_up": ([(50, 50, 3)] * 3, (64, 64)),
    "grey_375sq_to_64sq": ([(375, 375, 1)] * 3, (64, 64)),
    "ragged_to_64sq": ([(375, 375, 3), (480, 640, 3), (333, 500, 1), (50, 50, 3), (64, 64, 1), (1, 7, 3), (375, 375, 1)],
                       (64, 64)),
    "ragged_to_100x80": ([(375, 375, 3), (100, 80, 3), (77, 300, 1), (240, 60, 3)], (100, 80)),
}


def _images(shapes, seed):
    g = torch.Generator().manual_seed(seed)
    return [torch.randint(0, 256, s, generator=g, dtype=torch.uint8) for s in shapes]


def _aug(n, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.tensor([i % 2 for i in range(n)], dtype=torch.int32), torch.randint(-5, 6, (n, 2), generator=g,
                                                                                     dtype=torch.int32)


def _run(pipe, imgs, flip, shift):
    if len({tuple(t.shape) for t in imgs}) == 1:
        return pipe(torch.stack(imgs).cuda(), flip, shift)
    return pipe([t.cuda() for t in imgs], flip, shift)


@pytest.mark.parametrize("aug", [False, True], ids=["plain", "flip_shift"])
@pytest.mark.parametrize("name", list(CASES))
def test_rescale_matches_restatement(name, aug):
    shapes, size = CASES[name]
    imgs = _images(shapes, 11)
    flip, shift = _aug(len(imgs), 12) if aug else (None, None)
    got = _run(data.DevicePipeline(MEAN, STD, size=size), imgs, flip, shift)
    torch.cuda.synchronize()
    want = R.transform([t.numpy() for t in imgs], size, flip, shift, MEAN, STD)
    assert got.shape == want.shape
    err = ((got.double().cpu() - want) * torch.tensor(STD, dtype=torch.float64).view(1, 3, 1, 1)).abs().max().item()
    print(f"rescale {name} {'flip_shift' if aug else 'plain'}: max |error| on the [0, 1] scale {err:.3g}")
    assert err < TOL, err


def test_equal_size_is_bit_identical_to_image_pipeline():
    for C in (3, 1):
        imgs = _images([(64, 64, C)] * 5, 20 + C)
        flip, shift = _aug(5, 21)
        u8 = torch.stack(imgs).cuda()
        for f, s in ((None, None), (flip, shift)):
            a = data.DevicePipeline(MEAN, STD)(u8, f, s)
            b = data.DevicePipeline(MEAN, STD, size=(64, 64))(u8, f, s)
            assert torch.equal(a, b), C
    # the same per image inside a ragged batch (other images of other sizes around it)
    imgs = _images([(375, 375, 3), (64, 64, 3), (50, 50, 1), (64, 64, 1)], 22)
    flip, shift = _aug(4, 23)
    x = data.DevicePipeline(MEAN, STD, size=(64, 64))([t.cuda() for t in imgs], flip, shift)
    for i in (1, 3):
        ref = data.DevicePipeline(MEAN, STD)(imgs[i][None].cuda(), flip[i:i + 1], shift[i:i + 1])
        assert torch.equal(x[i:i + 1], ref), i


def test_two_calls_give_the_same_bits():
    imgs = [t.cuda() for t in _images(CASES["ragged_to_64sq"][0], 30)]
    flip, shift = _aug(len(imgs), 31)
    pipe = data.DevicePipeline(MEAN, STD, size=(64, 64))
    a = pipe(imgs, flip, shift)
    b = pipe(imgs, flip, shift)
    assert torch.equal(a, b)


def _pair(seed):
    mk = lambda: data.DevicePipeline(MEAN, STD, random_flip=True, max_shift=4, generator=torch.Generator().manual_seed(seed),
                                     size=(64, 64))
    return mk(), mk()


def test_resident_stimuli_batch_equals_direct_call():
    imgs = [t.numpy() for t in _images([(375, 375, 3), (500, 333, 3), (50, 50, 1), (375, 375, 3), (64, 64, 3)], 40)]
    imgs.append(imgs[2][:, :, 0])                                        # a grey stimulus given as [H, W]
    stim = data.ResidentStimuli(imgs)
    assert len(stim) == 6
    pa, pb = _pair(41)
    for idx in ([3, 0, 2, 2, 5], [1], [4, 3, 2, 1, 0, 5]):
        x = stim.batch(idx, pa)
        flip, shift = pb.draw(len(idx))
        y = pb([torch.from_numpy(np.ascontiguousarray(imgs[i].reshape(imgs[i].shape[0], imgs[i].shape[1], -1))).cuda()
                for i in idx], flip, shift)
        assert torch.equal(x, y), idx


def test_prefetcher_ragged_host_batches_equal_direct_call():
    shapes = [[(375, 375, 3), (50, 50, 1), (500, 333, 3)], [(64, 64, 3), (375, 375, 1)], [(100, 80, 3)] * 3]
    host = [[t.numpy() for t in _images(s, 50 + i)] for i, s in enumerate(shapes)]
    batches = [(b, {"fmri": torch.full((len(b), 7), float(i))}) for i, b in enumerate(host)]
    pa, pb = _pair(51)
    seen = 0
    for i, (x, ex) in enumerate(data.Prefetcher(batches, pa)):
        flip, shift = pb.draw(len(host[i]))
        y = pb([torch.from_numpy(a).cuda() for a in host[i]], flip, shift)
        assert torch.equal(x, y), i
        assert ex["fmri"].is_cuda and float(ex["fmri"][0, 0]) == float(i)
        seen += 1
    assert seen == 3
    # uniform host batches through a rescaling pipeline take the same path as a direct call
    u8 = _images([(375, 375, 3)] * 4, 52)
    pa, pb = _pair(53)
    x, _ = next(iter(data.Prefetcher([(torch.stack(u8), {})], pa)))
    flip, shift = pb.draw(4)
    assert torch.equal(x, pb(torch.stack(u8).cuda(), flip, shift))


def _errs(fn):
    before = L.launch_count()
    with pytest.raises(L.FmriError):
        fn()
    torch.cuda.synchronize()
    assert L.launch_count() == before


def test_argument_errors_raise_and_launch_nothing():
    buf = torch.zeros(375 * 375 * 3, dtype=torch.uint8, device="cuda")
    out = torch.empty(1, 3, 64, 64, device="cuda")
    ws = torch.empty(L.image_rescale_workspace(1), dtype=torch.uint8, device="cuda")
    call = lambda entries, o=out, w=ws, b=buf: L.image_rescale(b, L.image_src_table(entries), None, None, MEAN, STD, o, w)
    _errs(lambda: call([(0, 375, 375, 2)]))                                   # channels
    _errs(lambda: call([(0, 0, 375, 3)]))                                     # empty source
    _errs(lambda: call([(1, 375, 375, 3)]))                                   # past the end of the buffer
    _errs(lambda: call([(-8, 375, 375, 3)]))                                  # negative offset
    _errs(lambda: call([(0, 375, 375, 3)], w=ws[:8]))                         # workspace too small
    _errs(lambda: call([(0, 375, 375, 3)], w=ws[1:]))                         # workspace misaligned
    _errs(lambda: call([(0, 375, 375, 3), (0, 375, 375, 3)]))                 # two descriptors, one output image
    _errs(lambda: call([(0, 375, 375, 3)], o=torch.empty(1, 3, 64, 64, device="cuda", dtype=torch.float64)))
    _errs(lambda: call([(0, 375, 375, 3)], b=buf.cpu()))                      # host buffer
    big = torch.zeros(4000 * 4000 * 3, dtype=torch.uint8, device="cuda")      # source band larger than one CTA's smem
    _errs(lambda: call([(0, 4000, 4000, 3)], b=big))
    _errs(lambda: data.DevicePipeline(MEAN, STD)([buf.view(375, 375, 3)]))    # ragged input needs size=(H, W)
    _errs(lambda: data.DevicePipeline(MEAN, STD).rescale(buf, [(0, 375, 375, 3)]))
    _errs(lambda: data.DevicePipeline(MEAN, STD, size=(64, 64))([buf.view(375, 375, 3).cpu()]))


_REF = os.environ.get("FMRI_REFERENCE_ROOT")
_LOADER = os.path.join(_REF, "data_preprocessing", "data_loader.py") if _REF else None


def _real_skimage():
    try:
        import skimage
    except ImportError:
        return False
    return "script_harness" not in (getattr(skimage, "__file__", "") or "")


@pytest.mark.skipif(not (_LOADER and os.path.exists(_LOADER)) or not _real_skimage(),
                    reason="needs FMRI_REFERENCE_ROOT naming a checkout of the original project and real scikit-image")
def test_rescale_matches_reference_rescale(tmp_path):
    """The reference's own Rescale (data_preprocessing/data_loader.py) on BOLD5000-sized stimuli, run in a child process
    whose path holds only the reference tree (its `configs` package would clash with this repository's)."""
    imgs = [t.numpy() for t in _images([(375, 375, 3), (375, 375, 3)], 60)]
    np.save(tmp_path / "in.npy", np.stack(imgs))
    code = ("import sys, numpy as np; sys.path.insert(0, sys.argv[1]);"
            "from data_preprocessing.data_loader import Rescale;"
            "x = np.load(sys.argv[2]); t = Rescale((int(sys.argv[4]), int(sys.argv[4])));"
            "np.save(sys.argv[3], np.stack([np.asarray(t({'image': im, 'fmri': np.zeros(3620)})['image']) for im in x]))")
    for res in (100, 64):
        subprocess.run([sys.executable, "-c", code, _REF, str(tmp_path / "in.npy"), str(tmp_path / "out.npy"), str(res)],
                       check=True, cwd=_REF)
        ref = torch.from_numpy(np.load(tmp_path / "out.npy")).permute(0, 3, 1, 2)          # [N, 3, H, W] in [0, 1]
        got = data.DevicePipeline((0.0,) * 3, (1.0,) * 3, size=(res, res))(torch.stack([torch.from_numpy(a) for a in imgs]).cuda())
        err = (got.double().cpu() - ref.double()).abs().max().item()
        print(f"rescale vs the reference's Rescale at {res}: max |error| {err:.3g}")
        assert err < TOL, err
