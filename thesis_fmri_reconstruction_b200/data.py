"""The training step's left edge (SURVEY.md 8f-3): batches arrive from the host, the step wants normalised fp32 NCHW images
(and fp32 voxel vectors) resident in HBM.

Reference (all under /root/reference): the DataLoader workers decode and crop on the CPU, then apply per image
`RandomHorizontalFlip -> ToTensor (/255) -> GreyToColor -> Normalize(mean, std)` (train/train_vgan_stage1.py:161-171;
data_preprocessing/data_loader.py:374-400) or `Rescale -> RandomShift -> SampleToTensor -> Normalization` for the BOLD5000
stimuli (train/train_vgan_stage2.py:160-168; data_loader.py:93-111, 187-217), and the loop does `x.to(device)`
synchronously (train_vgan_stage1.py:322). Here the host ships the decoded uint8 pixels (4x fewer bytes than fp32) from
pinned memory on a copy stream while the previous step computes, and ONE kernel does the rest on the device:
fmri_image_pipeline (/255, grey -> RGB, flip, shift, normalisation) for pixels already at the training size, or, with
DevicePipeline(size=(H, W)), fmri_image_rescale, which first resizes native-resolution stimuli of any size as Rescale's
skimage.transform.resize does (Gaussian anti-aliasing + bilinear), or, with resample='bilinear' / 'bicubic',
fmri_image_resample, which resizes as PIL.Image.resize does (torchvision's Resize / CenterCrop / RandomResizedCrop on PIL
images, the COCO Stage-I loader's resize), byte for byte. JPEG decode stays on the host.

    pipe = DevicePipeline(mean=gan_cfg.mean, std=gan_cfg.std)
    for x, extras in Prefetcher(batches, pipe):       # batches yields (uint8 [B,H,W,C] tensor, dict of other host tensors)
        trainer.step(x, ...)

    pipe = DevicePipeline(mean, std, max_shift=5, size=(100, 100))
    stimuli = ResidentStimuli(images)                 # every stimulus in HBM once, at its native size
    x = stimuli.batch(indices, pipe)                  # no pixel crosses from the host per step

    coco = ResidentStimuli(images)                    # decoded images at their native sizes
    pipe = DevicePipeline(mean, std, random_flip=True, size=(64, 64), resample="bilinear")
    rrc = torchvision.transforms.RandomResizedCrop(64)
    crops = [rrc.get_params(torch.empty(1, h, w), rrc.scale, rrc.ratio) for _, h, w, _ in (coco.entries[i] for i in indices)]
    x = coco.batch(indices, pipe, crops=crops)       # RandomResizedCrop -> flip -> ToTensor -> Normalize on the device
"""
from __future__ import annotations

import torch

from . import lib as L


def pack_images(images, pin_memory=False):
    """One flat uint8 buffer holding uint8 [H, W, C] (C = 1 or 3) or [H, W] images back to back, on the images' device,
    and their (byte offset, H, W, C) descriptors."""
    ts = [im if isinstance(im, torch.Tensor) else torch.as_tensor(im) for im in images]
    if not ts:
        raise L.FmriError("pack_images needs at least one image")
    entries, off = [], 0
    for t in ts:
        if t.dtype != torch.uint8 or t.dim() not in (2, 3) or (t.dim() == 3 and t.shape[2] not in (1, 3)):
            raise L.FmriError(f"images must be uint8 [H, W] or [H, W, C] with C = 1 or 3, not {t.dtype} {tuple(t.shape)}")
        if t.device != ts[0].device:
            raise L.FmriError("pack_images: the images live on different devices")
        entries.append((off, t.shape[0], t.shape[1], t.shape[2] if t.dim() == 3 else 1))
        off += t.numel()
    dev = ts[0].device
    buf = torch.empty(off, dtype=torch.uint8, device=dev, pin_memory=pin_memory and dev.type == "cpu")
    torch.cat([t.reshape(-1) for t in ts], out=buf)
    return buf, entries


def resized_size(h, w, size):
    """Size (h', w') torchvision's Resize(size) gives an h x w image: `size` itself for an (h', w') pair, or for an int
    (or a 1-element sequence) the shorter side becomes size and the longer int(size * long / short), as in
    torchvision.transforms.functional._compute_resized_output_size without max_size."""
    if isinstance(size, (list, tuple)) and len(size) == 1:
        size = size[0]
    if isinstance(size, (list, tuple)):
        return int(size[0]), int(size[1])
    short, long = (w, h) if w <= h else (h, w)
    new_short, new_long = int(size), int(int(size) * long / short)
    return (new_long, new_short) if w <= h else (new_short, new_long)


def center_crop(h, w, size):
    """(top, left, height, width) of torchvision's CenterCrop(size) on an h x w image (size: int or (height, width)).
    A crop larger than the image, which torchvision pads, is refused."""
    ch, cw = (int(size), int(size)) if isinstance(size, int) else (int(size[0]), int(size[-1]))
    if ch > h or cw > w:
        raise L.FmriError(f"center crop {ch} x {cw} is larger than the {h} x {w} image (padding is not supported)")
    return int(round((h - ch) / 2.0)), int(round((w - cw) / 2.0)), ch, cw


def resample_windows(entries, size, resize=None, crops=None):
    """fmri_image_window tuples (offset, pitch, h, w, C, Hr, Wr, oy, ox) for the images `entries` ((byte offset, Hs, Ws, C)
    of dense HWC images) that produce size = (H, W) outputs as torchvision does on PIL images:
      crops[i] = (top, left, height, width) first crops image i (torchvision's crop, RandomResizedCrop.get_params or
      center_crop above), then the crop is resized to resized_size(h, w, resize), or to `size` when resize is None, and the
      centre H x W of that resize is kept (CenterCrop(size); the whole resize when resize is None)."""
    if crops is not None and len(crops) != len(entries):
        raise L.FmriError(f"{len(crops)} crop windows for {len(entries)} images")
    H, W = size
    out = []
    for i, (off, Hs, Ws, C) in enumerate(entries):
        top, left, h, w = (0, 0, Hs, Ws) if crops is None else (int(v) for v in crops[i])
        if top < 0 or left < 0 or h < 1 or w < 1 or top + h > Hs or left + w > Ws:
            raise L.FmriError(f"crop window {tuple(crops[i])} (top, left, height, width) leaves the {Hs} x {Ws} image {i}")
        Hr, Wr = (H, W) if resize is None else resized_size(h, w, resize)
        oy, ox = (0, 0) if resize is None else center_crop(Hr, Wr, (H, W))[:2]
        out.append((off + (top * Ws + left) * C, Ws * C, h, w, C, Hr, Wr, oy, ox))
    return out


class DevicePipeline:
    """uint8 [B, H, W, C] (C = 1 or 3) device tensor -> fp32 [B, 3, H, W], normalised, optionally flipped / shifted.
    With size=(H, W) the sources may have any size (a uniform [B, Hs, Ws, C] tensor or a list of per-image [Hs, Ws, C]
    device tensors) and are first resized to H x W as the reference's Rescale does (fmri_image_rescale); size=None keeps
    fmri_image_pipeline. resample='bilinear' or 'bicubic' (with size) resizes as PIL.Image.resize does instead
    (fmri_image_resample): to `size`, or, with resize=s, torchvision's Resize(s) followed by CenterCrop(size); per-image
    crop windows (crops=, see resample_windows) are taken first. The random draws use the torch RNG calls of the
    reference transforms' semantics (p = 0.5 flip per image; integer shifts uniform in [-max_shift, max_shift] per axis),
    made once per batch on the host."""

    def __init__(self, mean=(0.5, 0.5, 0.5), std=(0.5, 0.5, 0.5), random_flip=False, max_shift=0, generator=None,
                 size=None, resample=None, resize=None):
        self.mean, self.std = tuple(float(v) for v in mean), tuple(float(v) for v in std)
        self.random_flip, self.max_shift, self.gen = bool(random_flip), int(max_shift), generator
        self.size = None if size is None else (int(size[0]), int(size[1]))
        if resample is not None and (resample not in L.RESAMPLE_FILTERS or self.size is None):
            raise L.FmriError(f"resample={resample!r} needs size=(H, W) and one of {sorted(L.RESAMPLE_FILTERS)}")
        if resize is not None and resample is None:
            raise L.FmriError("resize= needs resample='bilinear' or 'bicubic'")
        self.resample, self.resize = resample, resize

    def draw(self, B):
        """Per-image augmentation parameters (host int32 tensors, or None): flip [B], shift_yx [B, 2]."""
        flip = shift = None
        if self.random_flip:
            flip = (torch.rand(B, generator=self.gen) < 0.5).to(torch.int32)
        if self.max_shift > 0:
            shift = torch.randint(-self.max_shift, self.max_shift + 1, (B, 2), generator=self.gen, dtype=torch.int32)
        return flip, shift

    @staticmethod
    def _params(t, device):
        return t.to(device, torch.int32, non_blocking=True).contiguous() if t is not None else None

    def __call__(self, u8, flip=None, shift_yx=None, out=None, crops=None):
        if self.size is not None and isinstance(u8, (list, tuple)):
            if not all(isinstance(t, torch.Tensor) and t.is_cuda for t in u8):
                raise L.FmriError("DevicePipeline expects device tensors (Prefetcher packs host images)")
            buf, entries = pack_images(u8)
            return self.rescale(buf, entries, flip, shift_yx, out, crops)
        if not isinstance(u8, torch.Tensor) or not u8.is_cuda or u8.dtype != torch.uint8 or u8.dim() != 4:
            raise L.FmriError("DevicePipeline expects a uint8 [B, H, W, C] tensor on the device")
        B, H, W, Cs = u8.shape
        if self.size is not None:
            n = H * W * Cs
            return self.rescale(u8.contiguous().view(-1), [(i * n, H, W, Cs) for i in range(B)], flip, shift_yx, out,
                                crops)
        if crops is not None:
            raise L.FmriError("crop windows need DevicePipeline(size=(H, W), resample='bilinear' or 'bicubic')")
        if out is None:
            out = torch.empty(B, 3, H, W, dtype=torch.float32, device=u8.device)
        L.image_pipeline(u8.contiguous(), self._params(flip, u8.device), self._params(shift_yx, u8.device), self.mean,
                         self.std, out)
        return out

    def rescale(self, buf, entries, flip=None, shift_yx=None, out=None, crops=None):
        """fp32 [N, 3, H, W] from the N images that `entries` ((byte offset, Hs, Ws, C) on the host) describe in the flat
        uint8 device buffer `buf`: resize to self.size (as Rescale does, or with resample= as PIL does, after the
        per-image crop windows `crops`), then shift / flip / GreyToColor / normalise."""
        if self.size is None:
            raise L.FmriError("rescale needs DevicePipeline(size=(H, W))")
        if crops is not None and self.resample is None:
            raise L.FmriError("crop windows need DevicePipeline(resample='bilinear' or 'bicubic')")
        dev = buf.device
        if out is None:
            out = torch.empty(len(entries), 3, *self.size, dtype=torch.float32, device=dev)
        flip, shift_yx = self._params(flip, dev), self._params(shift_yx, dev)
        if self.resample is None:
            ws = torch.empty(max(1, L.image_rescale_workspace(len(entries))), dtype=torch.uint8, device=dev)
            L.image_rescale(buf, L.image_src_table(entries), flip, shift_yx, self.mean, self.std, out, ws)
        else:
            table = L.image_window_table(resample_windows(entries, self.size, self.resize, crops))
            ws = torch.empty(max(1, L.image_resample_workspace(len(entries))), dtype=torch.uint8, device=dev)
            L.image_resample(buf, table, self.resample, flip, shift_yx, self.mean, self.std, out, ws)
        return out


class ResidentStimuli:
    """A stimulus set uploaded to HBM once, at its native sizes, as one uint8 buffer (BOLD5000's ~4.9 k stimuli at
    375 x 375 x 3 take about 2 GB); the descriptors stay on the host. batch(indices, pipeline) builds the descriptor
    table of those stimuli, draws the pipeline's flip / shift and resizes them on the device: after the upload a batch
    copies no pixels from the host, only 24 bytes of descriptor per image (48 with a resample= pipeline). `images`: a
    uint8 [N, H, W, C] tensor or a sequence of uint8 [H, W, C] / [H, W] arrays or tensors. `crops`: per-image
    (top, left, height, width) windows for a resample= pipeline, e.g. RandomResizedCrop.get_params draws."""

    def __init__(self, images, device="cuda"):
        host, self.entries = pack_images(list(images))
        self.buf = host.to(device)

    def __len__(self):
        return len(self.entries)

    def batch(self, indices, pipeline, out=None, crops=None):
        entries = [self.entries[int(i)] for i in indices]
        flip, shift = pipeline.draw(len(entries))
        return pipeline.rescale(self.buf, entries, flip, shift, out, crops)


class Prefetcher:
    """Double-buffered host -> device feed: while step i computes, batch i+1 is copied from pinned memory on a copy stream
    and run through the DevicePipeline on that stream. Iterating yields (images fp32 [B,3,H,W] on the device, extras dict on
    the device). `batches` yields (uint8 image tensor [B,H,W,C] on the host, dict of further host tensors, e.g. 'fmri');
    with DevicePipeline(size=(H, W)) the images may also be a list of per-image uint8 arrays of any sizes, which are
    packed into one pinned buffer and resized on the device."""

    def __init__(self, batches, pipeline, device="cuda"):
        self.it, self.pipe, self.dev = iter(batches), pipeline, torch.device(device)
        self.stream = torch.cuda.Stream()
        self._next = None
        self._stage()

    def _pin(self, t):
        return t if t.is_pinned() else t.pin_memory()

    def _stage(self):
        try:
            u8, extras = next(self.it)
        except StopIteration:
            self._next = None
            return
        ragged = isinstance(u8, (list, tuple))
        if ragged:
            u8, entries = pack_images(u8, pin_memory=True)
        flip, shift = self.pipe.draw(len(entries) if ragged else u8.shape[0])
        with torch.cuda.stream(self.stream):
            d8 = self._pin(u8).to(self.dev, non_blocking=True)
            x = self.pipe.rescale(d8, entries, flip, shift) if ragged else self.pipe(d8, flip, shift)
            ex = {k: self._pin(v).to(self.dev, non_blocking=True) for k, v in (extras or {}).items()}
            ev = torch.cuda.Event()
            ev.record(self.stream)
        self._next = (x, ex, ev, d8)

    def __iter__(self):
        return self

    def __next__(self):
        if self._next is None:
            raise StopIteration
        x, ex, ev, d8 = self._next
        cur = torch.cuda.current_stream()
        cur.wait_event(ev)
        for t in [x, d8] + list(ex.values()):
            t.record_stream(cur)
        self._stage()          # the next batch's copy + pipeline overlap this batch's compute
        return x, ex
