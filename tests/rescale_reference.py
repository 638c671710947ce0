"""fp64 restatement of the reference's BOLD5000 stimulus transform (data_preprocessing/data_loader.py Rescale -> RandomShift ->
SampleToTensor -> Normalization) for native-resolution uint8 stimuli. TEST INFRASTRUCTURE ONLY.

Rescale calls skimage.transform.resize(img, (H, W)) with its defaults. Neither scikit-image nor the reference is needed
here: resize() below restates what skimage >= 0.19 does for a uint8 image with those defaults (order 1, mode 'reflect',
anti_aliasing on when some axis downsamples, preserve_range False, clip True) in the scipy calls it makes:
    img_as_float                                  -> img / 255 in float64
    ndi.gaussian_filter(img, max(0, (f - 1) / 2), mode='mirror')   per axis f = in / out (channel axis: f = 1)
    ndi.zoom(img, 1 / f, order=1, mode='mirror', grid_mode=True)    samples at u = (o + 0.5) f - 0.5
    clip to [img.min(), img.max()]
It is a restatement, not the reference: tests/test_rescale_cpu.py compares it with real skimage when that is importable,
and tests/test_rescale_gpu.py compares the kernel with the reference's own Rescale when a checkout is named by
FMRI_REFERENCE_ROOT. The shift / flip / GreyToColor / normalisation after the resize are those of oracle.metrics.image_pipeline.
"""
import numpy as np
import torch
from scipy import ndimage as ndi


def resize(img_u8, out_hw):
    """uint8 [Hs, Ws] or [Hs, Ws, C] -> float64 [H, W] or [H, W, C] in [0, 1]."""
    a = np.asarray(img_u8).astype(np.float64) / 255.0
    out_shape = tuple(int(v) for v in out_hw) + a.shape[2:]
    factors = np.array(a.shape, dtype=np.float64) / np.array(out_shape, dtype=np.float64)
    x = a
    if np.any(factors > 1):
        x = ndi.gaussian_filter(a, np.maximum(0.0, (factors - 1) / 2), cval=0.0, mode="mirror")
    x = ndi.zoom(x, 1.0 / factors, order=1, mode="mirror", cval=0.0, grid_mode=True)
    assert x.shape == out_shape, (x.shape, out_shape)
    return np.clip(x, a.min(), a.max())


def transform(images, out_hw, flip=None, shift_yx=None, mean=(0.0,) * 3, std=(1.0,) * 3):
    """List of uint8 HWC (C = 1 or 3) or HW images -> float64 [N, 3, H, W]: resize, then the shift (edge replicate) and
    horizontal flip of the resized image, GreyToColor and (v - mean) / std."""
    H, W = (int(v) for v in out_hw)
    out = torch.empty(len(images), 3, H, W, dtype=torch.float64)
    ys, xs = torch.arange(H), torch.arange(W)
    for n, img in enumerate(images):
        r = torch.from_numpy(resize(img, (H, W)).reshape(H, W, -1)).permute(2, 0, 1).expand(3, H, W)
        yy, xx = ys, xs
        if flip is not None and int(flip[n]):
            xx = W - 1 - xx
        if shift_yx is not None:
            yy = (yy - int(shift_yx[n][0])).clamp(0, H - 1)
            xx = (xx - int(shift_yx[n][1])).clamp(0, W - 1)
        out[n] = r[:, yy][:, :, xx]
    m = torch.tensor(mean, dtype=torch.float64).view(1, 3, 1, 1)
    s = torch.tensor(std, dtype=torch.float64).view(1, 3, 1, 1)
    return (out - m) / s
